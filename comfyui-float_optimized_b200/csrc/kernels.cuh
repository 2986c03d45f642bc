// Non-GEMM kernels of the FMT sampling step.  All are bandwidth-trivial next to the weight stream; they exist to
// keep the data in the layout / precision the GEMMs want and to fuse what the reference does in separate torch ops.
//   AT = activation (GEMM operand) type: __nv_bfloat16 (FMT_MODE_BF16), bf16x3_t (FMT_MODE_BF16X3, gemm.cuh) or float (FMT_MODE_FP32_VALIDATE)
//   TT = AdaLN table type:               __nv_bfloat16                 float                                   or float
// Row layout of every activation matrix: m = branch * (B*N) + b * N + f, N = P + L frames (context first) - the
// same order the reference's batch-concatenated CFG forward uses (FMT.py:360-372).
#pragma once
#include "gemm.cuh"

namespace fmt {

// What one batch slot computes in one window: a window of its own clip (tensors of that clip alone, batch 1).  Every sampling entry
// point describes its windows this way: fmt_sample_clip's batch row b is slot b, fmt_velocity's clip b reads its explicit context
// through ctx and its [prev | current] conditions from win_start = P.
// An idle slot points at zeros, has r_d == nullptr, first_window == 1 and static emotion: it is computed and its output is dropped.
struct SlotArgs {
  const float* r_s;        // (W)
  const float* wa;         // (T_wa, A)
  const float* we;         // (T_we, E)
  const float* x0;         // (L, W) noise of this window of the clip
  float* r_d;              // (T_out, W), or nullptr for an idle slot
  int T_wa, T_we, T_out;
  int win_start;           // frame of wa / we that is this window's first current frame
  int first_window;        // 1: the clip starts in this window: zero context, whatever the slot ran before
  float a_scale, r_scale, e_scale;   // the clip's guidance
  int n_branches;          // 1, 3 or 4 (<= the plan's): the CFG branches the clip combines (slot_branch0)
  int out_start;           // frame of r_d that is this window's first current frame
  float* ctx;              // (P, W) the clip's motion context, read unless first_window and overwritten with this window's
                           // last P frames (fmt_sample_windows); nullptr: the context stays in the handle's per-slot state
  int we_dynamic;          // the clip's emotion: 0 static, we is (1, E) over every frame; 1 dynamic, we is (T_we, E) per frame
};

// The ODE schedule one slot runs in one window of fmt_sample_clips_ode / fmt_sample_windows_ode (the per-slot window graph).  In the
// slot-record buffer, the B SlotArgs of a window are followed by the B SlotOde of that window.  Plan evaluation e is the slot's step
// e / n_stages, stage e % n_stages while e < n_eval; from n_eval on the slot is idle: its x stays as it is.
struct SlotOde {
  const float* temb;       // (max(n_eval, 1), H) t-embedding of each of its evaluations (an idle slot: any valid row)
  const float* dt;         // (n_steps) step sizes
  int n_eval;              // n_steps * n_stages <= the plan's evaluation count
  int n_stages;            // 1..4
  float rk_a[16];          // a[g][j] at [g * 4 + j], zero-padded
  float rk_b[4];
};
__device__ __forceinline__ const SlotOde* slot_odes(const SlotArgs* slots, int B) { return reinterpret_cast<const SlotOde*>(slots + B); }

// First plan branch of a clip that combines nb of the plan's s_nb CFG branches.  Branches 1..3 of a 4-branch plan are
// [uncond | all | audio-only] with the null masks of a 3-branch plan (branch_nulls), so a 3-branch clip skips the truly-uncond
// branch; a 1-branch clip reads the `all` branch alone, the single conditional forward of FMT.py:400-401.
__host__ __device__ __forceinline__ int slot_branch0(int s_nb, int nb) { return nb == 1 ? (s_nb == 1 ? 0 : s_nb - 2) : s_nb - nb; }

// Per-window arguments, written to device memory by set_window_args so that the captured graph never changes.
struct WindowArgs {
  const SlotArgs* slots;   // (B) this window's slot records
};

struct ModelShape {
  int B, nb, N, P, L, W, A, E, H, Kc;   // Kc = padded c_embedder K (multiple of 64)
  unsigned null_a, null_r, null_e;      // bit br set = that condition is zeroed in branch br (FMT.py:360-392)
};

__global__ void set_window_args_kernel(WindowArgs* dst, WindowArgs v) { *dst = v; }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
// *p = v in the activation type; a bf16x3_t element writes its hi and lo parts where the pair layout puts them
template <typename T> __device__ __forceinline__ void store_act(T* p, float v) { *p = from_f32<T>(v); }
template <> __device__ __forceinline__ void store_act<bf16x3_t>(bf16x3_t* p, float v) {
  __nv_bfloat16* hp = split_hi(p);
  split_bf16(v, hp[0], hp[64]);
}

// ---------------------------------------------------------------------------------------------------------------
// Condition rows  [wr | wa | we | 0-pad]  for every (branch, clip, frame)   (FMT.py:312-333, nodes_adv.py:609-627,663-686)
// ---------------------------------------------------------------------------------------------------------------
template <typename AT>
__global__ void cond_gather_kernel(const WindowArgs* __restrict__ wargs, ModelShape s, const int* __restrict__ uidx, AT* __restrict__ cond) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const int rows = s.nb * s.B * s.N;
  // uidx != nullptr: block u builds the u-th DISTINCT condition row, the one token row uidx[u] sees (fmt_configure)
  const int row = uidx != nullptr ? uidx[blockIdx.x] : blockIdx.x;
  if (row >= rows) return;
  const int br = row / (s.B * s.N), b = (row / s.N) % s.B, f = row % s.N;
  const bool za = (s.null_a >> br) & 1, zr = (s.null_r >> br) & 1, ze = (s.null_e >> br) & 1;
  const bool ctx = f < s.P;
  const SlotArgs& sl = wargs->slots[b];   // the clip that slot b runs
  // frame of the clip this row looks at; replicate padding == clamp to the last available frame
  const int g = sl.win_start + f - s.P;
  AT* out = cond + static_cast<size_t>(blockIdx.x) * s.Kc;
  for (int j = threadIdx.x; j < s.Kc; j += blockDim.x) {
    float v = 0.f;
    if (j < s.W) {
      v = zr ? 0.f : sl.r_s[j];
    } else if (j < s.W + s.A) {
      const int k = j - s.W;
      // prev_wa is replicated un-nulled in every branch (FMT.py:366,388)
      if (ctx ? !sl.first_window : !za) v = sl.wa[static_cast<size_t>(min(g, sl.T_wa - 1)) * s.A + k];
    } else if (j < s.W + s.A + s.E) {
      const int k = j - s.W - s.A;
      if (!ze) {
        if (!sl.we_dynamic) v = sl.we[k];    // static emotion covers the context frames too (FMT.py:325-326)
        else if (!ctx || !sl.first_window) v = sl.we[static_cast<size_t>(min(g, sl.T_we - 1)) * s.E + k];
      }
    }
    store_act(out + j, v);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Timestep embedding (FMT.py:107-131), fp32 in every mode.  Runs once per plan.
// ---------------------------------------------------------------------------------------------------------------
__global__ void timestep_freq_kernel(const float* __restrict__ t, int n_eval, float* __restrict__ emb /* (n_eval, 256) */) {
  const int e = blockIdx.x, k = threadIdx.x;     // 128 threads
  const float neg_log = -9.210340371976184f;     // -ln(10000)
  const float freq = expf(neg_log * static_cast<float>(k) / 128.0f);
  const float arg = t[e] * freq;
  emb[e * 256 + k] = cosf(arg);
  emb[e * 256 + 128 + k] = sinf(arg);
}
// out[e, n] = act(sum_k W[n,k] * in[e,k] + b[n]); one warp per output element.
__global__ void small_linear_kernel(const float* __restrict__ in, const float* __restrict__ W, const float* __restrict__ b,
                                    float* __restrict__ out, int n_rows, int N, int K, int silu) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_rows * N) return;
  const int e = warp / N, n = warp % N;
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) acc = fmaf(W[static_cast<size_t>(n) * K + k], in[static_cast<size_t>(e) * K + k], acc);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    acc += b[n];
    out[static_cast<size_t>(e) * N + n] = silu ? acc / (1.f + expf(-acc)) : acc;
  }
}

// SiLU(c + t) of four elements: the AdaLN input of one condition row at one evaluation
__device__ __forceinline__ void silu_add4(const float4& c, const float4& t, float (&v)[4]) {
  v[0] = c.x + t.x; v[1] = c.y + t.y; v[2] = c.z + t.z; v[3] = c.w + t.w;
#pragma unroll
  for (int k = 0; k < 4; ++k) v[k] = v[k] / (1.f + expf(-v[k]));
}

// silu_c[(e*U + u), h] = SiLU(c_emb[u, h] + t_emb[e0 + e, h])      (FMT.py:335 then adaLN_modulation[0], :163-166)
template <typename AT>
__global__ void silu_cond_kernel(const float* __restrict__ c_emb, const float* __restrict__ t_emb, int e0, int U, int H,
                                 AT* __restrict__ out, size_t total) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  size_t i = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i >= total) return;
  const int h = static_cast<int>(i % H);
  const size_t row = i / H;
  const int u = static_cast<int>(row % U), e = static_cast<int>(row / U);
  const float4 c = *reinterpret_cast<const float4*>(c_emb + static_cast<size_t>(u) * H + h);
  const float4 t = *reinterpret_cast<const float4*>(t_emb + static_cast<size_t>(e0 + e) * H + h);
  float v[4];
  silu_add4(c, t, v);
  VecIO<AT, 4>::store(out + i, v);
}

// ---------------------------------------------------------------------------------------------------------------
// LayerNorm (eps 1e-6, no affine) + framewise modulate  x*(1+scale)+shift   (FMT.py:157,168-169,174-175,197)
// One warp per row; statistics in fp32 (two-pass).
// ---------------------------------------------------------------------------------------------------------------
template <typename AT, typename TT, int NV /* H / 128 float4 per lane */>
__global__ void lnmod_kernel(const float* __restrict__ X, int rows, int H, const TT* __restrict__ table, const int* __restrict__ urow,
                             long long ldt, long long shift_off, long long scale_off, AT* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* x = X + static_cast<size_t>(row) * H;
  const TT* trow = table + static_cast<size_t>(urow ? urow[row] : row) * ldt;
  float4 xv[NV];
  float sh[NV][4], sc[NV][4];
#pragma unroll
  for (int i = 0; i < NV; ++i) xv[i] = *reinterpret_cast<const float4*>(x + lane * 4 + i * 128);
#pragma unroll
  for (int i = 0; i < NV; ++i) {       // issued before the reductions so their latency overlaps the shuffles
    VecIO<TT, 4>::load(trow + shift_off + lane * 4 + i * 128, sh[i]);
    VecIO<TT, 4>::load(trow + scale_off + lane * 4 + i * 128, sc[i]);
  }
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) sum += (xv[i].x + xv[i].y) + (xv[i].z + xv[i].w);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum / static_cast<float>(H);
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float d0 = xv[i].x - mean, d1 = xv[i].y - mean, d2 = xv[i].z - mean, d3 = xv[i].w - mean;
    var += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) var += __shfl_xor_sync(0xffffffffu, var, o);
  const float rstd = rsqrtf(var / static_cast<float>(H) + 1e-6f);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    float v[4] = {(xv[i].x - mean) * rstd, (xv[i].y - mean) * rstd, (xv[i].z - mean) * rstd, (xv[i].w - mean) * rstd};
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = fmaf(v[k], 1.f + sc[i][k], sh[i][k]);
    VecIO<AT, 4>::store(out + static_cast<size_t>(row) * H + lane * 4 + i * 128, v);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Band-masked self-attention (FMT.py:15-19,69-88): row i attends j in [max(0,i-w), min(N-1,i+w)], scale hd^-1/2.
// One warp per (sequence, head, query row); the <= 2w+1 scores live in registers of the whole warp
// (dot products reduced with warp shuffles, softmax in fp32).  qkv columns: [q | k | v], each head-major.
// ---------------------------------------------------------------------------------------------------------------
template <typename AT, int VPL> struct RowVec;     // VPL consecutive elements of one lane, loaded with one instruction
template <> struct RowVec<float, 1> { static __device__ __forceinline__ void load(const float* p, float (&v)[1]) { v[0] = *p; } };
template <> struct RowVec<float, 2> { static __device__ __forceinline__ void load(const float* p, float (&v)[2]) { float2 t = *reinterpret_cast<const float2*>(p); v[0] = t.x; v[1] = t.y; } };
template <> struct RowVec<float, 4> { static __device__ __forceinline__ void load(const float* p, float (&v)[4]) { float4 t = *reinterpret_cast<const float4*>(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; } };
template <> struct RowVec<__nv_bfloat16, 1> { static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[1]) { v[0] = __bfloat162float(*p); } };
template <> struct RowVec<__nv_bfloat16, 2> { static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[2]) { __nv_bfloat162 t = *reinterpret_cast<const __nv_bfloat162*>(p); v[0] = __low2float(t); v[1] = __high2float(t); } };
template <> struct RowVec<__nv_bfloat16, 4> { static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[4]) { VecIO<__nv_bfloat16, 4>::load(p, v); } };

// OT: output type (bf16x3 mode reads fp32 q / k / v and writes the proj GEMM's pair operand)
template <typename AT, int VPL /* head_dim / 32 */, typename OT>
__global__ void band_attention_kernel(const AT* __restrict__ qkv, int n_seq, int N, int heads, int window, float scale,
                                      OT* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (gw >= n_seq * heads * N) return;
  const int i = gw % N, h = (gw / N) % heads, sq = gw / (N * heads);
  constexpr int hd = VPL * 32;
  const int Hd = heads * hd, ld = 3 * Hd;
  const AT* base = qkv + static_cast<size_t>(sq) * N * ld + h * hd + lane * VPL;
  float q[VPL];
  RowVec<AT, VPL>::load(base + static_cast<size_t>(i) * ld, q);
  const int j0 = max(0, i - window), j1 = min(N - 1, i + window);
  float mx = -INFINITY, den = 0.f, acc[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) acc[k] = 0.f;
  constexpr int KB = 5;                     // keys per batch: the default band (window 2) is one batch
  for (int jb = j0; jb <= j1; jb += KB) {
    float kv[KB][VPL], vv[KB][VPL], s[KB];
#pragma unroll
    for (int t = 0; t < KB; ++t) {          // all loads of the batch are issued before any use
      const int j = min(jb + t, j1);
      RowVec<AT, VPL>::load(base + static_cast<size_t>(j) * ld + Hd, kv[t]);
      RowVec<AT, VPL>::load(base + static_cast<size_t>(j) * ld + 2 * Hd, vv[t]);
    }
#pragma unroll
    for (int t = 0; t < KB; ++t) {
      float d = 0.f;
#pragma unroll
      for (int k = 0; k < VPL; ++k) d = fmaf(q[k], kv[t][k], d);
      s[t] = d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int t = 0; t < KB; ++t) s[t] += __shfl_xor_sync(0xffffffffu, s[t], o);
#pragma unroll
    for (int t = 0; t < KB; ++t) {          // online softmax over the band, fp32
      if (jb + t <= j1) {
        const float sc = s[t] * scale;
        const float nmx = fmaxf(mx, sc);
        const float corr = expf(mx - nmx), p = expf(sc - nmx);
        den = den * corr + p;
#pragma unroll
        for (int k = 0; k < VPL; ++k) acc[k] = fmaf(acc[k], corr, p * vv[t][k]);
        mx = nmx;
      }
    }
  }
  const float inv = 1.f / den;
  float o[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) o[k] = acc[k] * inv;
  OT* op = out + (static_cast<size_t>(sq) * N + i) * Hd + h * hd + lane * VPL;
  if constexpr (VPL == 4) VecIO<OT, 4>::store(op, reinterpret_cast<float(&)[4]>(o));
  else {
#pragma unroll
    for (int k = 0; k < VPL; ++k) store_act(op + k, o[k]);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Same attention for many sequences (>= 32 clips): one CTA per (sequence, head).  K and V of the head (N x head_dim bf16)
// are staged in shared memory once with coalesced 16-byte loads, so every qkv byte is read from L2 exactly once (the
// warp-per-row kernel above re-reads each K / V row for its 2w+1 neighbouring queries: 34 us vs ~10 us at 32 clips).
// ---------------------------------------------------------------------------------------------------------------
// Eight lanes share one query row (head_dim / 8 dims each, as 16-byte chunks interleaved so that a warp-wide LDS.128 is
// conflict-free), four rows per warp at a time: 3 shuffle steps per score instead of 5 and 4x fewer instructions per row than
// the 32-lanes-per-row mapping, which made this kernel issue-bound.
__device__ __forceinline__ void bf16x8_to_f32(const int4& t, float (&v)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
  for (int i = 0; i < 4; ++i) { v[2 * i] = __low2float(h[i]); v[2 * i + 1] = __high2float(h[i]); }
}
constexpr int ATTN_TILE_THREADS = 256;
template <int HD /* head_dim: 64 or 128 */>
__global__ void __launch_bounds__(ATTN_TILE_THREADS) band_attention_tile_kernel(const __nv_bfloat16* __restrict__ qkv, int N, int heads, int window, float scale,
                                                                                 __nv_bfloat16* __restrict__ out) {
  extern __shared__ __align__(16) uint8_t attn_smem[];
  constexpr int hd = HD, NCH = HD / 64;                         // 16-byte chunks per lane
  // Only K and V are staged (every row of them is read by 2w+1 queries); a query row is read once, straight from global memory, and
  // the whole K / V tile is requested in one batch (one L2 round trip instead of four).  Measured at 32 clips (768 CTAs): 21.0 us
  // with 128 threads and the online softmax, 15.9 us now; 80 registers x 256 threads put three CTAs on an SM (two waves), and what is
  // left is issue-bound: the bf16 -> fp32 conversions of the K / V chunks are half of the instructions of the band loop.
  __nv_bfloat16* sK = reinterpret_cast<__nv_bfloat16*>(attn_smem);
  __nv_bfloat16* sV = sK + static_cast<size_t>(N) * hd;
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const int h = blockIdx.x % heads, sq = blockIdx.x / heads;
  const int Hd = heads * hd, ld = 3 * Hd;
  const __nv_bfloat16* base = qkv + static_cast<size_t>(sq) * N * ld + h * hd;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sub = lane >> 3, dl = lane & 7;                     // row within the warp's group of 4, dim chunk
  const int rows_per_pass = (blockDim.x >> 5) * 4;
  // the query chunks of this lane's first row are requested together with the K / V tiles
  int4 q_raw[NCH];
  {
    const int ic0 = min(warp * 4 + sub, N - 1);
#pragma unroll
    for (int c = 0; c < NCH; ++c) q_raw[c] = *reinterpret_cast<const int4*>(base + static_cast<size_t>(ic0) * ld + c * 64 + dl * 8);
  }
  constexpr int CPR = hd / 8;                                  // 16-byte chunks per row
  constexpr int SB = 4;                                        // chunks per thread in flight: the whole tile is ONE round trip at N = 60
  for (int c0 = threadIdx.x; c0 < N * CPR; c0 += SB * blockDim.x) {
    int4 tk[SB], tv[SB];
#pragma unroll
    for (int b = 0; b < SB; ++b) {
      const int c = c0 + b * blockDim.x;
      if (c < N * CPR) {
        const int r = c / CPR, o = (c % CPR) * 8;
        tk[b] = *reinterpret_cast<const int4*>(base + static_cast<size_t>(r) * ld + Hd + o);
        tv[b] = *reinterpret_cast<const int4*>(base + static_cast<size_t>(r) * ld + 2 * Hd + o);
      }
    }
#pragma unroll
    for (int b = 0; b < SB; ++b) {
      const int c = c0 + b * blockDim.x;
      if (c < N * CPR) {
        const int r = c / CPR, o = (c % CPR) * 8;
        *reinterpret_cast<int4*>(sK + r * hd + o) = tk[b];
        *reinterpret_cast<int4*>(sV + r * hd + o) = tv[b];
      }
    }
  }
  __syncthreads();
  for (int i0 = warp * 4; i0 < N; i0 += rows_per_pass) {
    const int i = i0 + sub;
    const bool valid = i < N;
    const int ic = valid ? i : N - 1;
    float q[NCH][8];
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      bf16x8_to_f32(q_raw[c], q[c]);
#pragma unroll
      for (int k = 0; k < 8; ++k) q[c][k] *= scale;
    }
    {                                                            // next pass's query row: in flight while this one is computed
      const int in = min(i + rows_per_pass, N - 1);
#pragma unroll
      for (int c = 0; c < NCH; ++c) q_raw[c] = *reinterpret_cast<const int4*>(base + static_cast<size_t>(in) * ld + c * 64 + dl * 8);
    }
    const int j0 = max(0, ic - window), j1 = min(N - 1, ic + window);
    float mx = -INFINITY, den = 0.f, acc[NCH][8];
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[c][k] = 0.f;
    constexpr int KB = 5;
    // every lane of the warp runs the same number of key batches (shuffles are warp-wide): the widest band of the 4 rows
    const int nbatch = (2 * window + 1 + KB - 1) / KB;
    for (int bi = 0; bi < nbatch; ++bi) {
      const int jb = j0 + bi * KB;
      float s[KB];
#pragma unroll
      for (int t = 0; t < KB; ++t) {
        const int j = min(jb + t, j1);
        float d = 0.f;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          float kv[8];
          bf16x8_to_f32(*reinterpret_cast<const int4*>(sK + j * hd + c * 64 + dl * 8), kv);
#pragma unroll
          for (int k = 0; k < 8; ++k) d = fmaf(q[c][k], kv[k], d);
        }
        s[t] = d;
      }
#pragma unroll
      for (int o = 4; o > 0; o >>= 1)
#pragma unroll
        for (int t = 0; t < KB; ++t) s[t] += __shfl_xor_sync(0xffffffffu, s[t], o);
      // two-pass softmax over the batch (independent exponentials); batches are merged online only for bands wider than KB keys
      float bm = -INFINITY;
#pragma unroll
      for (int t = 0; t < KB; ++t) {
        if (jb + t > j1) s[t] = -INFINITY;
        bm = fmaxf(bm, s[t]);
      }
      if (bm == -INFINITY) continue;                            // a batch past this row's band (another row of the warp is wider)
      const float nmx = fmaxf(mx, bm);
      const float corr = __expf(mx - nmx);
      float p[KB], ps = 0.f;
#pragma unroll
      for (int t = 0; t < KB; ++t) { p[t] = __expf(s[t] - nmx); ps += p[t]; }
      den = fmaf(den, corr, ps);
      mx = nmx;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[c][k] *= corr;
#pragma unroll
        for (int t = 0; t < KB; ++t) {
          const int j = min(jb + t, j1);                        // p[t] = 0 past the band
          float vv[8];
          bf16x8_to_f32(*reinterpret_cast<const int4*>(sV + j * hd + c * 64 + dl * 8), vv);
#pragma unroll
          for (int k = 0; k < 8; ++k) acc[c][k] = fmaf(p[t], vv[k], acc[c][k]);
        }
      }
    }
    if (valid) {
      const float inv = __fdividef(1.f, den);
      __nv_bfloat16* op = out + (static_cast<size_t>(sq) * N + i) * Hd + h * hd + dl * 8;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        int4 t;
        __nv_bfloat162* hp = reinterpret_cast<__nv_bfloat162*>(&t);
#pragma unroll
        for (int k = 0; k < 4; ++k) hp[k] = __floats2bfloat162_rn(acc[c][2 * k] * inv, acc[c][2 * k + 1] * inv);
        *reinterpret_cast<int4*>(op + c * 64) = t;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Classifier-free-guidance combine (FMT.py:375-379,396-399), incremental form exactly as the reference writes it.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float cfg_combine(const float* __restrict__ V, size_t idx, size_t branch_stride, int nb, float a, float r,
                                             float e) {
  if (nb == 1) return V[idx];
  if (nb == 3) {
    const float u = V[idx], c = V[idx + branch_stride], ao = V[idx + 2 * branch_stride];
    return u + a * (ao - u) + e * (c - ao);
  }
  const float tu = V[idx], u = V[idx + branch_stride], c = V[idx + 2 * branch_stride], ao = V[idx + 3 * branch_stride];
  return tu + r * (u - tu) + a * (ao - u) + e * (c - ao);
}

// The same selection for the persistent kernels' COMB, which hold the plan's branches in vb[0..3]: the scales and branch count of
// the clip in slot b, and vb shifted so that vb[0] is its first branch (constant register indices).
__device__ __forceinline__ void slot_guidance(const SlotArgs* slots, int s_nb, int b, float (&vb)[4], int& nb, float& a, float& r, float& e) {
  const SlotArgs& sl = slots[b];
  nb = __ldg(&sl.n_branches);
  a = __ldg(&sl.a_scale); r = __ldg(&sl.r_scale); e = __ldg(&sl.e_scale);
  const int br0 = slot_branch0(s_nb, nb);
  if (br0 >= 1) { vb[0] = vb[1]; vb[1] = vb[2]; vb[2] = vb[3]; }
  if (br0 >= 2) { vb[0] = vb[1]; vb[1] = vb[2]; }
}

// Every producer of an ODE state also writes the x-embedder operand rows of that state (replicated over the CFG
// branches, FMT.py:363): ax[(br, b, P + f), :] = bf16(y[b, f, :]).  Context rows are written once per window.
template <typename AT>
__device__ __forceinline__ void store_ax(const ModelShape& s, AT* __restrict__ ax, int b, int f_full, int j, float v) {
  if constexpr (std::is_same<AT, bf16x3_t>::value) {
    __nv_bfloat16 hi, lo;
    split_bf16(v, hi, lo);
    for (int br = 0; br < s.nb; ++br) {
      __nv_bfloat16* hp = split_hi(ax + ((static_cast<size_t>(br) * s.B + b) * s.N + f_full) * s.W + j);
      hp[0] = hi; hp[64] = lo;
    }
  } else {
    const AT t = from_f32<AT>(v);
    for (int br = 0; br < s.nb; ++br) ax[((static_cast<size_t>(br) * s.B + b) * s.N + f_full) * s.W + j] = t;
  }
}

// The ODE updates of torchdiffeq's fixed-grid solvers, shared by the plan's kernels and the per-slot schedule kernels so that both
// round alike: Euler y0 + dt * v, and the Runge-Kutta stage / final combination y0 + dt * sum_j c[j] * k_j over the first n_k stages
__device__ __forceinline__ float euler_update(const float* dt, float v, const float* y0) { return fmaf(*dt, v, *y0); }
__device__ __forceinline__ float rk_update(const float (&c)[4], const float* k, size_t k_stride, size_t i, int n_k,
                                           const float* dt, const float* y0) {
  float acc = 0.f;
  for (int j = 0; j < n_k; ++j)
    if (c[j] != 0.f) acc = fmaf(c[j], k[j * k_stride + i], acc);
  return fmaf(*dt, acc, y0[i]);
}

// mode 0: v_full[b, f, :] = combined, all N frames (fmt_velocity)
// mode 1: k_out[b, f-P, :] = combined, current frames only (RK stage derivative)
// mode 2: y[b, f-P, :] += dt * combined   (fused CFG + Euler update, torchdiffeq euler: y1 = y0 + dt*f(t0,y0))
template <typename AT>
__global__ void cfg_combine_kernel(const WindowArgs* __restrict__ wargs, ModelShape s, const float* __restrict__ V, int mode,
                                   float* __restrict__ dst, const float* __restrict__ dt_ptr, AT* __restrict__ ax) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t per_branch = static_cast<size_t>(s.B) * s.N * s.W;
  if (i >= per_branch) return;
  const int j = static_cast<int>(i % s.W);
  const int f = static_cast<int>((i / s.W) % s.N), b = static_cast<int>(i / (static_cast<size_t>(s.W) * s.N));
  if (mode != 0 && f < s.P) return;
  const SlotArgs& sl = wargs->slots[b];   // the clip's own scales and branches
  const int nb = sl.n_branches;
  const float v = cfg_combine(V, i + slot_branch0(s.nb, nb) * per_branch, per_branch, nb, sl.a_scale, sl.r_scale, sl.e_scale);
  if (mode == 0) dst[i] = v;
  else {
    const size_t o = (static_cast<size_t>(b) * s.L + (f - s.P)) * s.W + j;
    if (mode == 1) dst[o] = v;
    else {
      const float y = euler_update(dt_ptr, v, dst + o);
      dst[o] = y;
      store_ax<AT>(s, ax, b, f, j, y);
    }
  }
}

// y_out = y0 + dt * sum_j coef[j] * k_j   (explicit Runge-Kutta stage / final combination); also refreshes ax
template <typename AT>
__global__ void rk_combine_kernel(ModelShape s, const float* __restrict__ y0, float* __restrict__ y_out, const float* __restrict__ k,
                                  size_t n, size_t k_stride, int n_k, float c0, float c1, float c2, float c3,
                                  const float* __restrict__ dt_ptr, AT* __restrict__ ax) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float c[4] = {c0, c1, c2, c3};
  const float y = rk_update(c, k, k_stride, i, n_k, dt_ptr, y0);
  y_out[i] = y;
  const int j = static_cast<int>(i % s.W), f = static_cast<int>((i / s.W) % s.L), b = static_cast<int>(i / (static_cast<size_t>(s.W) * s.L));
  store_ax<AT>(s, ax, b, s.P + f, j, y);
}

// Window prologue: x_state <- the slot's x0, context rows <- prev_x or the slot's own ctx (zero in the first window,
// nodes_adv.py:591), ax <- [context | x0]
template <typename AT>
__global__ void init_window_kernel(const WindowArgs* __restrict__ wargs, ModelShape s, float* __restrict__ x_state,
                                   float* __restrict__ prev_x_state, AT* __restrict__ ax) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<size_t>(s.B) * s.N * s.W) return;
  const int j = static_cast<int>(i % s.W), f = static_cast<int>((i / s.W) % s.N), b = static_cast<int>(i / (static_cast<size_t>(s.W) * s.N));
  const SlotArgs& sl = wargs->slots[b];
  float v;
  if (f < s.P) {
    const size_t o = (static_cast<size_t>(b) * s.P + f) * s.W + j;
    if (sl.first_window) { v = 0.f; prev_x_state[o] = 0.f; }
    else if (sl.ctx != nullptr) v = sl.ctx[static_cast<size_t>(f) * s.W + j];
    else v = prev_x_state[o];
  } else {
    const size_t o = (static_cast<size_t>(b) * s.L + (f - s.P)) * s.W + j;
    v = sl.x0[static_cast<size_t>(f - s.P) * s.W + j];
    x_state[o] = v;
  }
  store_ax<AT>(s, ax, b, f, j, v);
}
// Window epilogue: the slot's r_d[out_start + f] <- x_state for the frames below its T_out (an idle slot writes nothing), prev_x
// (and the slot's ctx) <- last P frames (nodes_adv.py:659-668,690-692)
__global__ void finalize_window_kernel(const WindowArgs* __restrict__ wargs, ModelShape s, const float* __restrict__ x_state,
                                       float* __restrict__ prev_x_state) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<size_t>(s.B) * s.L * s.W) return;
  const int j = static_cast<int>(i % s.W), f = static_cast<int>((i / s.W) % s.L), b = static_cast<int>(i / (static_cast<size_t>(s.W) * s.L));
  const float v = x_state[i];
  const SlotArgs& sl = wargs->slots[b];
  const int g = sl.out_start + f;
  if (sl.r_d != nullptr && g < sl.T_out) sl.r_d[static_cast<size_t>(g) * s.W + j] = v;
  if (f >= s.L - s.P) {
    const int c = f - (s.L - s.P);
    prev_x_state[(static_cast<size_t>(b) * s.P + c) * s.W + j] = v;
    if (sl.ctx != nullptr) sl.ctx[static_cast<size_t>(c) * s.W + j] = v;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Per-slot ODE schedules (the per-slot window graph): every slot reads its own SlotOde; the arithmetic is the plan kernels'
// ---------------------------------------------------------------------------------------------------------------
// silu_c[(e*U + u), h] = SiLU(c_emb[u, h] + t_emb[h]) with the t-embedding of evaluation e0 + e of the schedule of the slot that
// condition row u belongs to.  uidx: the token row of every distinct row (nullptr: row u); no distinct row spans two slots here.
template <typename AT>
__global__ void silu_cond_sched_kernel(const WindowArgs* __restrict__ wargs, ModelShape s, const float* __restrict__ c_emb,
                                       const int* __restrict__ uidx, int e0, int U, AT* __restrict__ out, size_t total) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const int H = s.H;
  size_t i = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i >= total) return;
  const int h = static_cast<int>(i % H);
  const size_t row = i / H;
  const int u = static_cast<int>(row % U), e = e0 + static_cast<int>(row / U);
  const int tok = uidx != nullptr ? uidx[u] : u;
  const SlotOde& o = slot_odes(wargs->slots, s.B)[(tok / s.N) % s.B];
  const float* t_emb = o.temb + (e < o.n_eval ? static_cast<size_t>(e) * H : 0);
  const float4 c = *reinterpret_cast<const float4*>(c_emb + static_cast<size_t>(u) * H + h);
  const float4 t = *reinterpret_cast<const float4*>(t_emb + h);
  float v[4];
  silu_add4(c, t, v);
  VecIO<AT, 4>::store(out + i, v);
}

// Before plan evaluation e: y_g = y0 + dt * sum_j a[g][j] k_j for every slot that is at a stage g > 0 of its own schedule (also
// refreshes ax); a slot at stage 0 already holds x in ax
template <typename AT>
__global__ void sched_stage_kernel(const WindowArgs* __restrict__ wargs, ModelShape s, const float* __restrict__ x_state,
                                   float* __restrict__ y_stage, const float* __restrict__ k, size_t n, int e, AT* __restrict__ ax) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int j = static_cast<int>(i % s.W), f = static_cast<int>((i / s.W) % s.L), b = static_cast<int>(i / (static_cast<size_t>(s.W) * s.L));
  const SlotOde& o = slot_odes(wargs->slots, s.B)[b];
  const int G = o.n_stages, g = e % G;
  if (e >= o.n_eval || g == 0) return;
  const float c[4] = {o.rk_a[g * 4], o.rk_a[g * 4 + 1], o.rk_a[g * 4 + 2], o.rk_a[g * 4 + 3]};
  const float y = rk_update(c, k, n, i, g, o.dt + e / G, x_state);
  y_stage[i] = y;
  store_ax<AT>(s, ax, b, s.P + f, j, y);
}

// After plan evaluation e: every slot that is at an evaluation of its own schedule combines its CFG branches (as
// cfg_combine_kernel does) and takes its Euler step (one-stage solvers), or stores k_g and, after its last stage, takes
// x += dt * sum_j b[j] k_j (as rk_combine_kernel does).  k holds up to four stages of n elements each.
template <typename AT>
__global__ void sched_combine_kernel(const WindowArgs* __restrict__ wargs, ModelShape s, const float* __restrict__ V, int e,
                                     float* __restrict__ x_state, float* k, size_t n, AT* __restrict__ ax) {
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t per_branch = static_cast<size_t>(s.B) * s.N * s.W;
  if (i >= per_branch) return;
  const int j = static_cast<int>(i % s.W);
  const int f = static_cast<int>((i / s.W) % s.N), b = static_cast<int>(i / (static_cast<size_t>(s.W) * s.N));
  if (f < s.P) return;
  const SlotArgs* slots = wargs->slots;
  const SlotOde& o = slot_odes(slots, s.B)[b];
  if (e >= o.n_eval) return;
  const SlotArgs& sl = slots[b];
  const int nb = sl.n_branches;
  const float v = cfg_combine(V, i + slot_branch0(s.nb, nb) * per_branch, per_branch, nb, sl.a_scale, sl.r_scale, sl.e_scale);
  const size_t oi = (static_cast<size_t>(b) * s.L + (f - s.P)) * s.W + j;
  const int G = o.n_stages, g = e % G;
  const float* dt = o.dt + e / G;
  float y;
  if (G == 1) {
    y = euler_update(dt, v, x_state + oi);
  } else {
    k[g * n + oi] = v;
    if (g < G - 1) return;
    const float c[4] = {o.rk_b[0], o.rk_b[1], o.rk_b[2], o.rk_b[3]};
    y = rk_update(c, k, n, oi, G, dt, x_state);
  }
  x_state[oi] = y;
  store_ax<AT>(s, ax, b, f, j, y);
}

// fp32 -> bf16 weight packing (with optional K padding)
__global__ void pack_weight_kernel(const float* __restrict__ src, int rows, int K, __nv_bfloat16* __restrict__ dst, int Kpad) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<size_t>(rows) * Kpad) return;
  const int k = static_cast<int>(i % Kpad);
  const size_t r = i / Kpad;
  dst[i] = __float2bfloat16_rn(k < K ? src[r * K + k] : 0.f);
}
// fp32 -> bf16 of a dense activation matrix, 8 elements per thread (two 16-byte loads, one 16-byte store): the HBM-bound pass in
// front of the audio-projection GEMM (n % 8 == 0)
__global__ void f32_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, size_t n8) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n8; i += stride) {
    const float4 a = __ldcs(reinterpret_cast<const float4*>(src) + 2 * i), b = __ldcs(reinterpret_cast<const float4*>(src) + 2 * i + 1);
    uint4 t;
    t.x = pack_bf16x2(a.x, a.y); t.y = pack_bf16x2(a.z, a.w); t.z = pack_bf16x2(b.x, b.y); t.w = pack_bf16x2(b.z, b.w);
    reinterpret_cast<uint4*>(dst)[i] = t;
  }
}

// fp32 -> bf16x3 pairs, 4 elements per thread: the weights (once per handle, from Linear::w32) and the audio-projection input.
// Rows must hold a multiple of 64 elements (n4 = elements / 4).
__global__ void f32_to_split_kernel(const float* __restrict__ src, bf16x3_t* __restrict__ dst, size_t n4) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 a = __ldcs(reinterpret_cast<const float4*>(src) + i);
    const float v[4] = {a.x, a.y, a.z, a.w};
    VecIO<bf16x3_t, 4>::store(dst + 4 * i, v);
  }
}

// Audio projection tail (FLOAT.py:338-342: Linear -> LayerNorm(affine, eps) -> SiLU): one warp per row of the GEMM output.
__global__ void ln_silu_kernel(const float* __restrict__ y, long long rows, int N, const float* __restrict__ g, const float* __restrict__ b,
                               float eps, float* __restrict__ out) {
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* yr = y + row * N;
  float sum = 0.f;
  for (int c = lane * 4; c < N; c += 128) {
    const float4 v = *reinterpret_cast<const float4*>(yr + c);
    sum += (v.x + v.y) + (v.z + v.w);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum / static_cast<float>(N);
  float var = 0.f;
  for (int c = lane * 4; c < N; c += 128) {
    const float4 v = *reinterpret_cast<const float4*>(yr + c);
    const float d0 = v.x - mean, d1 = v.y - mean, d2 = v.z - mean, d3 = v.w - mean;
    var += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) var += __shfl_xor_sync(0xffffffffu, var, o);
  const float rstd = rsqrtf(var / static_cast<float>(N) + eps);
  for (int c = lane * 4; c < N; c += 128) {
    const float4 v = *reinterpret_cast<const float4*>(yr + c);
    const float4 gg = __ldg(reinterpret_cast<const float4*>(g + c)), bb = __ldg(reinterpret_cast<const float4*>(b + c));
    float t[4] = {(v.x - mean) * rstd * gg.x + bb.x, (v.y - mean) * rstd * gg.y + bb.y, (v.z - mean) * rstd * gg.z + bb.z,
                  (v.w - mean) * rstd * gg.w + bb.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) t[k] = t[k] / (1.f + expf(-t[k]));          // SiLU
    *reinterpret_cast<float4*>(out + row * N + c) = make_float4(t[0], t[1], t[2], t[3]);
  }
}

__global__ void pad_weight_f32_kernel(const float* __restrict__ src, int rows, int K, float* __restrict__ dst, int Kpad) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<size_t>(rows) * Kpad) return;
  const int k = static_cast<int>(i % Kpad);
  const size_t r = i / Kpad;
  dst[i] = k < K ? src[r * K + k] : 0.f;
}

}  // namespace fmt
