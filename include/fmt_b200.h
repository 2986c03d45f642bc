/*
 * fmt_b200.h - C ABI of the B200-native FMT motion-latent sampler (libfmt_b200.so).
 *
 * This is the drop-in boundary for ONE path of set-soft/ComfyUI-FLOAT_Optimized: the Flow-Matching-
 * Transformer ODE sampling loop.  Reference interfaces replaced (paths relative to the reference repo):
 *
 *   src/nodes/nodes_adv.py:545-694   _perform_ode_sampling_loop  -> fmt_sample_clip
 *   src/nodes/models/float/FLOAT.py:172-253  FLOAT.sample        -> fmt_sample_clip (static emotion, 3 branches)
 *   src/nodes/models/float/FMT.py:342-401   forward_with_cfv     -> fmt_velocity
 *   src/nodes/models/float/FMT.py:277-340   forward              -> (inside fmt_velocity / fmt_sample_clip)
 *   torchdiffeq.odeint fixed-grid solvers (nodes_adv.py:658)     -> FmtPlan (Butcher tableau) + fmt_sample_clip
 *
 * Conventions
 *   - plain C types only; every tensor is a dense row-major fp32 array.
 *   - pointers are DEVICE pointers unless the struct says `location = FMT_LOC_HOST`.
 *   - every call returns 0 on success, <0 on error (fmt_last_error() gives the message); no C++ exception
 *     crosses this boundary.  A handle is bound to one CUDA device and is not thread-safe.
 *   - all work is enqueued on the given cudaStream_t (passed as void*); calls do not synchronise unless
 *     documented (host-located outputs synchronise the stream before returning).
 *   - there is NO CPU fallback: on a machine without an sm_100 device fmt_create fails.
 */
#ifndef FMT_B200_H
#define FMT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FMT_API __attribute__((visibility("default")))
#define FMT_ABI_VERSION 2

typedef struct FmtHandle FmtHandle;

/* Mirror of the BaseOptions fields the FMT reads (src/nodes/options/base_options.py:10-60). */
typedef struct FmtDims {
  int32_t dim_w;            /* motion latent width (512)            */
  int32_t dim_a;            /* audio latent width (512)             */
  int32_t dim_e;            /* emotion classes (7)                  */
  int32_t dim_h;            /* hidden size (1024)                   */
  int32_t depth;            /* FMT blocks (8)                       */
  int32_t num_heads;        /* attention heads (8)                  */
  int32_t mlp_hidden;       /* int(dim_h * mlp_ratio) (4096)        */
  int32_t num_prev_frames;  /* context frames P (10)                */
  int32_t frames_per_clip;  /* window length L = int(wav2vec_sec*fps) (50) */
  int32_t attention_window; /* band half-width (2), FMT.py:15-19    */
} FmtDims;

/* Order of the fp32 weight pointers handed to fmt_create (nn.Linear layout: (out,in) row-major).
 * Global tensors first, then FMT_W_PER_BLOCK pointers per block. */
enum {
  FMT_W_X_W = 0,      /* x_embedder.proj.weight (H, dim_w)            */
  FMT_W_X_B,          /* x_embedder.proj.bias   (H)                   */
  FMT_W_T0_W,         /* t_embedder.mlp.0.weight (H, 256)             */
  FMT_W_T0_B,
  FMT_W_T2_W,         /* t_embedder.mlp.2.weight (H, H)               */
  FMT_W_T2_B,
  FMT_W_C_W,          /* c_embedder.weight (H, dim_w+dim_a+dim_e), columns [wr | wa | we] */
  FMT_W_C_B,
  FMT_W_POS,          /* pos_embed (P+L, H)                           */
  FMT_W_DEC_ADA_W,    /* decoder.adaLN_modulation.1.weight (2H, H)    */
  FMT_W_DEC_ADA_B,
  FMT_W_DEC_W,        /* decoder.linear.weight (dim_w, H)             */
  FMT_W_DEC_B,
  FMT_W_NUM_GLOBAL
};
enum {
  FMT_WB_QKV_W = 0,   /* blocks.i.attn.qkv.weight (3H, H), rows [q | k | v], head-major */
  FMT_WB_QKV_B,
  FMT_WB_PROJ_W,      /* blocks.i.attn.proj.weight (H, H)             */
  FMT_WB_PROJ_B,
  FMT_WB_FC1_W,       /* blocks.i.mlp.fc1.weight (mlp_hidden, H)      */
  FMT_WB_FC1_B,
  FMT_WB_FC2_W,       /* blocks.i.mlp.fc2.weight (H, mlp_hidden)      */
  FMT_WB_FC2_B,
  FMT_WB_ADA_W,       /* blocks.i.adaLN_modulation.1.weight (6H, H): shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp */
  FMT_WB_ADA_B,
  FMT_W_PER_BLOCK
};

enum { FMT_LOC_DEVICE = 0, FMT_LOC_HOST = 1 };
enum { FMT_MODE_BF16 = 0,       /* bf16 tcgen05/TMA GEMMs, fp32 accumulate / residual / LN / softmax / ODE state */
       FMT_MODE_FP32_VALIDATE = 1, /* same kernels' epilogues + fp32 SIMT GEMMs: the 1e-4 parity mode         */
       FMT_MODE_BF16X3 = 2         /* tcgen05 GEMMs on split operands x = hi + lo (two bf16 each), Ah.Wh + Ah.Wl + Al.Wh in fp32:
                                      fp32-class accuracy (the 1e-4 gates) on the tensor pipe; AdaLN tables, QKV and every
                                      non-GEMM step in fp32.  The first plan in this mode packs the weights once more
                                      (4 bytes per weight: 627 MB for the FMT).  Plans of <= 256 token rows run one kernel per
                                      op (the persistent window kernels are bf16-only).                                    */ };

#define FMT_MAX_STAGES 4

/* What forward_with_cfv batches and how the ODE grid is walked.  One plan = one captured CUDA graph. */
typedef struct FmtPlan {
  int32_t batch;          /* clips B                                                                        */
  int32_t n_branches;     /* 1: all scales == 1 (FMT.py:400-401); 3: default CFG; 4: include_r_cfg (:380-399) */
  int32_t we_dynamic;     /* 0: we is (B,1,E) broadcast over all P+L frames; 1: we is (B,T,E).  The emotion mode of
                             fmt_sample_clip, fmt_velocity and of the clip / window sets without per-clip modes; no
                             graph depends on it, so a plan that differs only in it is not re-captured            */
  int32_t mode;           /* FMT_MODE_*                                                                      */
  int32_t n_steps;        /* ODE steps S = nfe-1 (torchdiffeq fixed grid: nfe points)                        */
  int32_t n_stages;       /* explicit RK stages per step (euler 1, midpoint 2, heun2 2, heun3 3, rk4 4)      */
  const float* t_eval;    /* HOST (n_steps*n_stages): time of every function evaluation, fp32               */
  const float* dt;        /* HOST (n_steps): t[i+1]-t[i] in fp32                                            */
  const float* rk_a;      /* HOST (n_stages*n_stages) strictly lower-triangular: y_i = y0 + dt*sum_j a[i][j]*k_j */
  const float* rk_b;      /* HOST (n_stages): y1 = y0 + dt*sum_j b[j]*k_j                                    */
} FmtPlan;

typedef void (*fmt_progress_fn)(int32_t window_index, int32_t n_windows, void* user);

/* One sampler call = _perform_ode_sampling_loop (nodes_adv.py:545-694). */
typedef struct FmtClip {
  int32_t location;       /* FMT_LOC_DEVICE or FMT_LOC_HOST for ALL pointers below                           */
  const float* r_s;       /* (B, dim_w)  reference-identity latent wr                                        */
  const float* wa;        /* (B, T_wa, dim_a) audio latents                                                  */
  const float* we;        /* (B, T_we, dim_e) with T_we == 1 (static) or the dynamic length                  */
  const float* noise;     /* (n_windows, B, L, dim_w): x0 of every window, drawn by the caller in window order
                             (torch.randn(B,L,dim_w, generator) per window, nodes_adv.py:606)                */
  float* r_d;             /* out (B, audio_num_frames, dim_w)                                                */
  int32_t T_wa;
  int32_t T_we;
  int32_t audio_num_frames;
  float a_cfg_scale, r_cfg_scale, e_cfg_scale;
  fmt_progress_fn progress; /* optional: called on the host after each window is enqueued (ProgressBar tick, nodes_adv.py:688) */
  void* progress_user;
} FmtClip;

/* Many independent clips in one call (fmt_sample_clips): clip i is what fmt_sample_clip gives for it alone (batch 1) with its noise.
 * Every pointer is a DEVICE pointer; the arrays themselves are host arrays of n_clips entries. */
typedef struct FmtClipSet {
  int32_t n_clips;
  const float* const* r_s;          /* [i]: (1, dim_w)                                                                     */
  const float* const* wa;           /* [i]: (1, T_wa[i], dim_a)                                                            */
  const float* const* we;           /* [i]: (1, T_we[i], dim_e); T_we[i] == 1 (static) or > 1 (dynamic), per clip's emotion mode    */
  const float* const* noise;        /* [i]: (n_win_i, L, dim_w), n_win_i = ceil(audio_num_frames[i] / L): x0 of each of its windows */
  float* const* r_d;                /* [i]: out (1, audio_num_frames[i], dim_w); only these frames are written                  */
  const int32_t* T_wa;
  const int32_t* T_we;
  const int32_t* audio_num_frames;
  float a_cfg_scale, r_cfg_scale, e_cfg_scale;   /* shared by every clip                                                      */
  fmt_progress_fn progress;         /* optional: called on the host after each window of the schedule is enqueued (index, makespan) */
  void* progress_user;
} FmtClipSet;

/* Guidance of every clip of a FmtClipSet (fmt_sample_clips_guided): host arrays of n_clips entries.  n_branches[i] is the
 * reference's rule for clip i's scales and include_r_cfg (FMT.py:346,380,400): 1 when every scale is 1, else 3, or 4 with the
 * r guidance term.  A clip with fewer branches than the plan combines only its own: a 3-branch clip in a 4-branch plan the
 * branches [uncond | all | audio-only], a 1-branch clip the `all` branch alone. */
typedef struct FmtClipGuidance {
  const float* a_cfg_scale;
  const float* r_cfg_scale;
  const float* e_cfg_scale;
  const int32_t* n_branches;        /* 1, 3 or 4, <= plan.n_branches; a 1-branch plan takes 1-branch clips only */
} FmtClipGuidance;

/* One window of each of n_streams streams (fmt_sample_windows): a stream is a clip whose audio arrives in pieces, run one window per
 * call.  Every pointer is a DEVICE pointer; the arrays themselves are host arrays of n_streams entries.  Window w of a stream reads
 * wa / we frames [w*L - P, (w+1)*L) and writes its frames [w*L, w*L + n_out); the buffers below start at its first context frame. */
typedef struct FmtWindowSet {
  int32_t n_streams;                /* 1 <= n_streams <= plan.batch; stream i runs in slot i, slots n_streams.. are idle            */
  const float* const* r_s;          /* [i]: (1, dim_w)                                                                           */
  const float* const* wa;           /* [i]: (T_wa[i], dim_a) from frame w*L - P (frame 0 in a first window); frames beyond T_wa[i]
                                       are the last frame repeated, as in a clip's last window                                  */
  const float* const* we;           /* [i]: static (1, dim_e), or dynamic (T_we[i], dim_e) from the same frame as wa (the stream's
                                       emotion mode: plan.we_dynamic, or its entry of fmt_sample_window_set's we_dynamic)       */
  const float* const* x0;           /* [i]: (L, dim_w) noise of this window                                                      */
  float* const* ctx;                /* [i]: (P, dim_w) in / out: the last P frames of the stream's previous window (not read in a
                                       first window); receives this window's last P frames                                       */
  float* const* r_d;                /* [i]: out (n_out[i], dim_w): the window's first n_out[i] frames                             */
  const int32_t* T_wa;              /* frames of wa[i]; the window's first current frame (P, or 0 in a first window) must be one  */
  const int32_t* T_we;              /* 1 (static) or the frames of we[i] (dynamic), likewise                                     */
  const int32_t* n_out;             /* 1 <= n_out[i] <= L                                                                        */
  const int32_t* first_window;      /* 1: the stream's window 0: zero context                                                   */
} FmtWindowSet;

/* The ODE schedule of every clip of a FmtClipSet or stream of a FmtWindowSet (fmt_sample_clips_ode, fmt_sample_windows_ode): host
 * arrays of n_clips / n_streams entries, each entry laid out as the FmtPlan fields of the same names (HOST arrays).  Clip i runs
 * n_steps[i] * n_stages[i] evaluations per window, at most the plan's n_steps * n_stages, with 1..FMT_MAX_STAGES stages; its result
 * is what a plan with its own schedule gives for it.  n_steps[i] = 0 (nfe 1) returns the noise. */
typedef struct FmtClipOde {
  const int32_t* n_steps;
  const int32_t* n_stages;
  const float* const* t_eval;       /* [i]: (n_steps[i] * n_stages[i]) times of its evaluations                                  */
  const float* const* dt;           /* [i]: (n_steps[i])                                                                          */
  const float* const* rk_a;         /* [i]: (n_stages[i] * n_stages[i])                                                           */
  const float* const* rk_b;         /* [i]: (n_stages[i])                                                                         */
} FmtClipOde;

/* One evaluation of forward_with_cfv (FMT.py:342-401) on explicit window inputs - tests and ncu. */
typedef struct FmtEval {
  const float* x;         /* (B, L, dim_w)                     */
  const float* prev_x;    /* (B, P, dim_w)                     */
  const float* wa;        /* (B, L, dim_a)                     */
  const float* prev_wa;   /* (B, P, dim_a)                     */
  const float* we;        /* (B, 1|L, dim_e) per plan.we_dynamic */
  const float* prev_we;   /* (B, P, dim_e) or NULL when static  */
  const float* r_s;       /* (B, dim_w)                        */
  float* v_out;           /* out (B, P+L, dim_w): the CFG-combined model output, context rows included */
  int32_t eval_index;     /* which t_eval[] entry of the plan  */
  float a_cfg_scale, r_cfg_scale, e_cfg_scale;
} FmtEval;

FMT_API int32_t fmt_abi_version(void);
FMT_API const char* fmt_last_error(void);

/* Packs the reference's fp32 weights into resident bf16 (and keeps fp32 for the validation mode and the bf16x3 packing).
 * weight_ptrs: FMT_W_NUM_GLOBAL + depth*FMT_W_PER_BLOCK pointers, all at `location`. */
FMT_API int32_t fmt_create(const FmtDims* dims, const void* const* weight_ptrs, int32_t n_ptrs, int32_t location,
                           int32_t device, FmtHandle** out);
FMT_API int32_t fmt_destroy(FmtHandle* h);

/* Sizes the workspace, computes the timestep embeddings of every evaluation and (re)captures the window
 * graph.  Cheap when the plan equals the current one. */
FMT_API int32_t fmt_configure(FmtHandle* h, const FmtPlan* plan, void* stream);
FMT_API int64_t fmt_workspace_bytes(const FmtHandle* h);

/* Whole clip: all windows, chained on the device through prev_x / prev_wa / prev_we. */
FMT_API int32_t fmt_sample_clip(FmtHandle* h, const FmtClip* clip, void* stream);

/* Host-only (no device work): the slot schedule of fmt_sample_clips.  n_windows[i] >= 1 is the window count of clip i.  Clips are
 * taken in order of window count, descending (ties in input order); each goes to the slot that is free first (ties: lowest slot)
 * and starts there at its own window 0 in the window that slot becomes free.  n_slots = 0 picks the smallest slot count <= 256
 * whose schedule finishes in max(n_windows) windows (256 if none does); n_slots > 0 schedules on exactly that many slots.
 * Fills slot_out[i] / start_out[i] (may be NULL) and *makespan_out (may be NULL, the number of windows the call runs) and
 * returns the slot count, < 0 on bad arguments. */
FMT_API int32_t fmt_clip_schedule(int32_t n_clips, const int32_t* n_windows, int32_t n_slots, int32_t* slot_out, int32_t* start_out,
                                  int32_t* makespan_out);

/* Many clips of different lengths in one call, on plan.batch slots refilled as clips finish (device pointers only).  plan.batch
 * must equal fmt_clip_schedule(n_slots = 0)'s slot count for these clips' window counts; each clip must pass fmt_sample_clip's
 * checks with batch 1.  The window graph of the plan is replayed once per window of the schedule (its makespan).
 * Every clip uses the set's scales and plan.n_branches: fmt_sample_clips_guided with that guidance. */
FMT_API int32_t fmt_sample_clips(FmtHandle* h, const FmtClipSet* set, void* stream);

/* fmt_sample_clips with each clip's own guidance; the set's a/r/e_cfg_scale are not read.  Clip i's result depends only on its
 * own inputs and guidance and on the plan.  Returns -1 if an n_branches[i] is not 1, 3 or 4 or exceeds plan.n_branches, or if a
 * 1-branch plan gets a clip with more than one branch. */
FMT_API int32_t fmt_sample_clips_guided(FmtHandle* h, const FmtClipSet* set, const FmtClipGuidance* guidance, void* stream);

/* One window of each stream of the set, with each stream's own guidance (n_streams entries; as in fmt_sample_clips_guided), stream i
 * in slot i.  The call replays a window graph of fmt_occupancy_slots(plan.batch, n_streams) slots, captured the first time a call
 * needs it (a plan whose window graph is the persistent window kernel replays its one graph of plan.batch slots).  A stream's window
 * computes what the same window of fmt_sample_clips computes for the whole clip, bit for bit, whichever graph it runs in.  Returns -1
 * on bad arguments. */
FMT_API int32_t fmt_sample_windows(FmtHandle* h, const FmtWindowSet* set, const FmtClipGuidance* guidance, void* stream);

/* fmt_sample_clips_guided / fmt_sample_windows with each clip / stream on its own ODE schedule (ode == NULL: exactly the call without
 * it).  They run a second window graph of the plan, captured on first use: every evaluation of the plan, in which a slot whose clip
 * needs fewer runs its own ones first and then stays idle (its x is kept, its rows are computed and dropped), with one kernel per op
 * at any row count (plans of <= 256 token rows too, which the plan's graph runs in the persistent window kernel).  The t-embeddings
 * of each distinct schedule are computed the first time it is seen and kept in the handle.  Return -1 if a clip needs more
 * evaluations than the plan or more than FMT_MAX_STAGES stages, or on the checks of the calls without ode. */
FMT_API int32_t fmt_sample_clips_ode(FmtHandle* h, const FmtClipSet* set, const FmtClipGuidance* guidance, const FmtClipOde* ode, void* stream);
FMT_API int32_t fmt_sample_windows_ode(FmtHandle* h, const FmtWindowSet* set, const FmtClipGuidance* guidance, const FmtClipOde* ode,
                                       void* stream);

/* The general entries the five calls above are written with.  guidance == NULL (clip sets only): the set's a/r/e_cfg_scale and
 * plan.n_branches for every clip; ode == NULL: the plan's schedule (the plan's window graph); we_dynamic == NULL: plan.we_dynamic for
 * every clip / stream, else a HOST array of n_clips / n_streams entries, 0 (static emotion: T_we[i] == 1) or 1 (dynamic: T_we[i] > 1
 * for a clip, with the coverage checks of its mode).  Clips of both modes share one call and the plan's window graphs: the condition
 * rows they share do not depend on the mode (fmt_debug_condition_rows_slots).  Clip i's result is what a call whose every clip has
 * clip i's mode gives for it on the same plan.  Returns -1 on a mode other than 0 / 1 or a T_we that does not match it, or on the
 * checks of the calls above. */
FMT_API int32_t fmt_sample_clip_set(FmtHandle* h, const FmtClipSet* set, const FmtClipGuidance* guidance, const FmtClipOde* ode,
                                    const int32_t* we_dynamic, void* stream);
FMT_API int32_t fmt_sample_window_set(FmtHandle* h, const FmtWindowSet* set, const FmtClipGuidance* guidance, const FmtClipOde* ode,
                                      const int32_t* we_dynamic, void* stream);

/* Host-only (no device work): the slots of the window graph a call of fmt_sample_window_set with n_ready streams runs on a plan of
 * plan_slots slots - the smallest of 1, 2, 4, ... (the powers of two below plan_slots) and plan_slots that is >= n_ready.  Returns
 * < 0 unless 1 <= n_ready <= plan_slots <= 256. */
FMT_API int32_t fmt_occupancy_slots(int32_t plan_slots, int32_t n_ready);
/* Slots of the window graph the last sampling call replayed (0 before the first). */
FMT_API int32_t fmt_last_window_slots(const FmtHandle* h);

/* Single CFG-combined model evaluation (device pointers). */
FMT_API int32_t fmt_velocity(FmtHandle* h, const FmtEval* ev, void* stream);

/* Counters for bench.py: kernels this library launched (graph nodes included) since the last reset. */
FMT_API int64_t fmt_launch_count(const FmtHandle* h, int32_t reset);
/* Number of kernel nodes in the captured window graph (0 before fmt_configure). */
FMT_API int32_t fmt_graph_kernel_nodes(const FmtHandle* h);
/* The same for the per-slot window graph of fmt_sample_clips_ode / fmt_sample_windows_ode (0 before its first call on this plan). */
FMT_API int32_t fmt_ode_graph_kernel_nodes(const FmtHandle* h);

/* Persistent window kernel (plans with <= 256 token rows, bf16): > 0 = id of the bounded spin that tripped (the kernel traps instead
 * of hanging the GPU), whatever ran since; else -1 = not in use for the current plan, or the last sampling call ran the per-slot
 * window graph (one kernel per op); 0 = in use and healthy. */
FMT_API int32_t fmt_window_kernel_status(const FmtHandle* h);

/* With FMT_WIN_TRACE=1 in the environment at fmt_configure: copies the per-CTA barrier stamps of the last window,
 * [cta][barrier][arrive, pass] in SM clocks, into `out` (HOST); returns the element count (call with NULL to size). */
FMT_API int64_t fmt_debug_window_trace(const FmtHandle* h, int64_t* out, int64_t max_elems);
/* Host-only (no device work): which token rows (branch, clip, frame) of forward_with_cfv's batched forward (FMT.py:360-392) see the
 * same condition row [wr | wa | we] - the AdaLN tables hold one row per DISTINCT condition row.  Fills urow[n_branches * batch *
 * n_frames] (may be NULL) with the distinct-row index of every token row and returns the number of distinct rows, < 0 on bad
 * arguments. */
FMT_API int32_t fmt_debug_condition_rows(int32_t n_branches, int32_t batch, int32_t n_frames, int32_t n_prev, int32_t we_dynamic,
                                         int32_t* urow_out);
/* The same with per_slot = 1 for the per-slot window graph, whose distinct rows never span two slots (batch - 1 more rows in 4-branch
 * plans: the truly-unconditional current frames are one row per slot). */
FMT_API int32_t fmt_debug_condition_rows_ode(int32_t n_branches, int32_t batch, int32_t n_frames, int32_t n_prev, int32_t we_dynamic,
                                             int32_t per_slot, int32_t* urow_out);
/* The same with slot b's emotion mode we_dynamic[b] (HOST, batch entries): the map the keys of every slot's own mode give.  The
 * sampler uses the map of plan.we_dynamic for every mix; this entry shows that the map is the same. */
FMT_API int32_t fmt_debug_condition_rows_slots(int32_t n_branches, int32_t batch, int32_t n_frames, int32_t n_prev,
                                               const int32_t* we_dynamic, int32_t per_slot, int32_t* urow_out);

/* ---- audio projection in front of the sampler (SURVEY.md 8f rank 2) ----
 * Replaces the nn.Sequential(Linear(in_dim, dim_w), LayerNorm(dim_w), SiLU) that FloatApplyAudioProjection runs
 * (src/nodes/nodes_vadv.py:147-198; module built in src/nodes/models/float/FLOAT.py:338-342 and
 * src/nodes/nodes_vadv_loader.py:228-257): wa = SiLU(LayerNorm(x W^T + b)).  in_dim = 9216 (12 stacked wav2vec layers) or 768. */
typedef struct FmtProj FmtProj;
FMT_API int32_t fmt_proj_create(int32_t in_dim, int32_t out_dim, const float* linear_w /* (out_dim, in_dim) */, const float* linear_b,
                                const float* ln_w, const float* ln_b, float ln_eps, int32_t location, int32_t device, FmtProj** out);
FMT_API int32_t fmt_proj_destroy(FmtProj* p);
/* x (rows, in_dim) fp32 -> out (rows, out_dim) fp32, both at `location` (FMT_LOC_HOST synchronises the stream).  mode as in FmtPlan. */
FMT_API int32_t fmt_proj_apply(FmtProj* p, const float* x, int64_t rows, float* out, int32_t mode, int32_t location, void* stream);
FMT_API int64_t fmt_proj_launch_count(const FmtProj* p, int32_t reset);

/* ---- diagnostic entry points (unit tests of the kernels; not used by the node) ---- */
/* out[M,N] (fp32) = A[M,K] (bf16 bits) @ W[N,K]^T (bf16 bits) + bias[N], through the tcgen05/TMA GEMM. */
FMT_API int32_t fmt_debug_gemm_bf16(const void* A, const void* W, const float* bias, float* out, int32_t M, int32_t N,
                                    int32_t K, int32_t block_n, void* stream);
/* `iters` back-to-back launches of one GEMM variant (bf16 output); block_n as above, 512 / 1024 = CTA-pair kernel. */
FMT_API int32_t fmt_debug_gemm_bench(const void* A, const void* W, const float* bias, float* out, int32_t M, int32_t N,
                                     int32_t K, int32_t block_n, int32_t iters, void* stream);
/* out[M,N] (fp32) = A[M,K] (fp32) @ W[N,K]^T (fp32) + bias[N] through the bf16x3 GEMM of FMT_MODE_BF16X3: the operands are split
 * into hi / lo bf16 pairs on the device (K % 64 == 0).  block_n as in fmt_debug_gemm_bf16: 64 / 128 / 256 single-CTA kernel,
 * 512 / 1024 CTA-pair kernel, 0 = the choice the sampler makes. */
FMT_API int32_t fmt_debug_gemm_bf16x3(const float* A, const float* W, const float* bias, float* out, int32_t M, int32_t N,
                                      int32_t K, int32_t block_n, void* stream);
/* `iters` back-to-back launches of one bf16x3 GEMM variant, fp32 output.  A (M, 2K) and W (N, 2K) are bf16 bits already in the pair
 * layout: every 64-column K block of hi = bf16(x) followed by the same block of lo = bf16(x - hi). */
FMT_API int32_t fmt_debug_gemm_bench_bf16x3(const void* A, const void* W, const float* bias, float* out, int32_t M, int32_t N,
                                            int32_t K, int32_t block_n, int32_t iters, void* stream);
/* Same through the fp32 SIMT GEMM used by FMT_MODE_FP32_VALIDATE (A, W fp32). */
FMT_API int32_t fmt_debug_gemm_fp32(const float* A, const float* W, const float* bias, float* out, int32_t M, int32_t N,
                                    int32_t K, void* stream);

/* Fused GEMM epilogues of the FMT step (FMT.py:171-176), applied to acc = A . W^T + bias:
 *   STORE     out = acc
 *   GELU      out = GELU_tanh(acc)
 *   POS       out = acc + pos[(m % frames) * N + n]
 *   GATE_RES  out[m, n] += gate[urow[m] * ldg + gate_off + n] * acc   (out fp32; urow NULL = identity)  */
enum { FMT_EPI_STORE = 0, FMT_EPI_GELU = 1, FMT_EPI_POS = 2, FMT_EPI_GATE_RES = 3 };

/* One GEMM of fmt_debug_gemm_epilogue.  Every pointer is a DEVICE pointer. */
typedef struct FmtDebugGemm {
  int32_t mode;           /* FMT_MODE_*: bf16 tcgen05, fp32 SIMT or bf16x3 tcgen05 GEMM                                  */
  int32_t kind;           /* FMT_EPI_*                                                                                    */
  int32_t M, N, K;
  int32_t block_n;        /* 0 = the sampler's choice; 64 / 128 / 256 single-CTA kernel, 512 / 1024 CTA-pair kernel (not fp32) */
  int32_t ksplit;         /* K slices of the CTA-pair kernel (1 = none; > 1: GATE_RES only, K >= 64 * ksplit)              */
  int32_t ldo;            /* row stride of out in elements (>= N)                                                         */
  int32_t out_f32;        /* 1: out is fp32; 0: the mode's activation type (bf16 bits, bf16x3 pairs or fp32).  GATE_RES: 1 */
  int32_t frames;         /* POS: rows of pos                                                                             */
  const float* A;         /* (M, K) fp32, rounded to bf16 (bf16) or split into pairs (bf16x3) on the device               */
  const float* W;         /* (N, K) fp32, likewise                                                                        */
  const float* bias;      /* (N) or NULL                                                                                  */
  void* out;              /* (M, ldo); bf16x3 pairs: ldo % 64 == 0 and 256-byte aligned (gemm.cuh)                        */
  const float* pos;       /* POS: (frames, N)                                                                             */
  const void* gate;       /* GATE_RES: the AdaLN table in the mode's table type (bf16 bits in bf16 mode, else fp32)       */
  const int32_t* urow;    /* GATE_RES: table row of every output row, or NULL                                            */
  int64_t ldg;            /* GATE_RES: table row stride in elements                                                      */
  int64_t gate_off;       /* GATE_RES: column of the gate's first element                                                */
} FmtDebugGemm;

/* One GEMM with a fused epilogue, dispatched exactly as the sampler dispatches its GEMMs in `mode`. */
FMT_API int32_t fmt_debug_gemm_epilogue(const FmtDebugGemm* g, void* stream);
/* LayerNorm (eps 1e-6, no affine) + modulate of the sampler: out[r] = LN(X[r]) * (1 + table[t + scale_off]) + table[t + shift_off]
 * with t = (urow ? urow[r] : r) * ldt.  X (rows, H) fp32, H in {128, 256, 512, 1024}; table in the mode's table type; out (rows, H)
 * in the mode's activation type. */
FMT_API int32_t fmt_debug_lnmod(int32_t mode, const float* X, int32_t rows, int32_t H, const void* table, const int32_t* urow,
                                int64_t ldt, int64_t shift_off, int64_t scale_off, void* out, void* stream);
/* Band attention of the sampler (FMT.py:15-19,69-88): qkv (n_seq, N, 3 * heads * hd) in the mode's table type, columns [q | k | v]
 * head-major; out (n_seq, N, heads * hd) in the mode's activation type.  hd in {32, 64, 128}.  variant 0 = the sampler's choice,
 * 1 = one warp per query row, 2 = one CTA per (sequence, head) with K / V in shared memory (bf16 mode, hd 64 or 128, K and V of a
 * head within 48 KB); returns -1 for a variant that cannot run these arguments. */
FMT_API int32_t fmt_debug_band_attention(int32_t mode, const void* qkv, int32_t n_seq, int32_t N, int32_t heads, int32_t hd,
                                         int32_t window, void* out, int32_t variant, void* stream);

/* Row-wise stages of the persistent window kernels (bf16 mode), run by the kernels' own stage functions:
 *   ROW   mode 0: X = Pacc + bias + pos[frame];  mode 1: X += gate * (Pacc + bias);  then A1 = bf16(LN(X) (1 + scale) + shift), Pacc <- 0
 *         (window kernel with zero_qkv: the QKV accumulator rows <- 0 as well)
 *   ATTN  A2 = bf16(band attention of QKVacc + bias) (flow kernel: QKV buffer `parity`, the valid rows of the other buffer <- 0)
 *   GELU  Hm = bf16(GELU_tanh(Hacc + bias)), Hacc <- 0
 *   COMB  CFG combine of Vacc + bias (decoder bias), then Euler or stage `stage` of an explicit Runge-Kutta step `step`: kbuf[stage],
 *         x_state at the last stage, ax = bf16(y) in every branch; Vacc <- 0
 * Token rows: n_branches x batch sequences of n_frames, the first n_prev of them context frames.  Row layouts:
 *   flow kernel    chunks of chunk_rows (32 / 64) rows that never straddle a sequence: RP = chunks x chunk_rows padded rows, NPs =
 *                  chunk_rows x ceil(n_frames / chunk_rows) per sequence.  X, Pacc, Hacc (RP, .); QKVacc two buffers (RP, 3H);
 *                  Vacc (n_branches, batch, NPs, W); A1 / A2 / Hm [chunk][K block][chunk_rows][64] with the 16-byte XOR swizzle.
 *   window kernel  R = n_branches x batch x n_frames <= 256 rows, Rp = R rounded up to 64: X, Pacc, QKVacc, Hacc (R, .); Vacc
 *                  (n_branches, batch, n_frames, W); A1 / A2 / Hm [K block][Rp][64] with the same swizzle.
 * Every pointer is a DEVICE pointer except slot_branches / slot_scales. */
enum { FMT_STAGE_ROW = 0, FMT_STAGE_ATTN = 1, FMT_STAGE_GELU = 2, FMT_STAGE_COMB = 3 };

typedef struct FmtDebugStage {
  int32_t kind;           /* FMT_STAGE_*                                                                                 */
  int32_t grid;           /* CTAs, 0 = one per SM (flow kernel: at least one per chunk)                                 */
  int32_t chunk_rows;     /* flow kernel: 32 or 64 (window kernel: ignored)                                             */
  int32_t n_branches, batch, n_frames, n_prev;
  int32_t H, heads, window, mlp_hidden, W;   /* H in {128, 256, 512, 1024}; ATTN: H / heads in {32, 64, 128}          */
  int32_t row_mode, zero_qkv, parity;
  int32_t n_stages, stage, step;             /* COMB: stages of the solver (1 = Euler), the stage and step it runs       */
  int64_t ldt;            /* ROW: AdaLN table row stride (elements)                                                     */
  int64_t gate_off, shift_off, scale_off;    /* ROW: table columns of gate (mode 1), shift and scale                    */
  float a_scale, r_scale, e_scale;           /* COMB: guidance of every clip without slot_branches                      */
  float rk_a[16], rk_b[4];                   /* COMB: a[g][j] at [g * n_stages + j], b[j]                               */
  float *X, *Pacc, *QKVacc, *Hacc, *Vacc;
  void *A1, *A2, *Hm, *ax;                   /* bf16                                                                     */
  const void* table;      /* ROW: bf16 AdaLN table (rows, ldt)                                                          */
  const int32_t* urow;    /* ROW, flow kernel: table row of every token row, or NULL                                    */
  const float* bias;      /* ROW: (H); ATTN: (3H); GELU: (mlp_hidden); COMB: (W)                                        */
  const float* pos;       /* ROW mode 0: (n_frames, H)                                                                   */
  float *x_state, *kbuf;  /* COMB: (batch, n_frames - n_prev, W) and n_stages of those                                  */
  const float* ddt;       /* COMB: step sizes, at least step + 1                                                         */
  const int32_t* slot_branches;              /* COMB, HOST or NULL: per clip 1, 3 or 4 branches (<= n_branches)         */
  const float* slot_scales;                  /* COMB, HOST (batch, 3): per clip a, r, e scales (with slot_branches)     */
} FmtDebugStage;

/* One stage kind of the dataflow window kernel (flow.cuh) over every chunk. */
FMT_API int32_t fmt_debug_flow_stage(const FmtDebugStage* d, void* stream);
/* One stage kind of the barrier-stepped window kernel (window.cuh, split-K schedule) over every row. */
FMT_API int32_t fmt_debug_window_stage(const FmtDebugStage* d, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FMT_B200_H */
