// Dataflow window kernel for the weight-streaming regime (a few clips per GPU): successor of the barrier-stepped kernel in
// window.cuh.  One launch of one CTA per SM runs EVERY model evaluation of a sampling window, but no stage ever waits for
// the whole grid:
//
//   * The token rows are cut into CHUNKS of CH (32 or 64) rows that never straddle a sequence (a CFG branch of a clip).  Chunks
//     are independent dependency chains - only band attention looks at the neighbouring chunk of the same sequence and only
//     the CFG combine looks at the other branches - so while one chain waits for an L2 round trip the SM works on another.
//   * Every (evaluation, stage, chunk) has its own release counter in global memory.  A producer bumps it (red.release.gpu)
//     once its part is visible, a consumer polls exactly the counters it depends on (ld.acquire.gpu): the weight-stationary
//     split-K GEMM of a chunk starts as soon as the SIMT stage before it has finished THAT chunk, the SIMT stage of a chunk as
//     soon as every K slice of THAT chunk has been reduced.  Nothing is ever reset: counters are per instance.
//   * A CTA is two engines that walk the same stage list independently.  GEMM engine: warp 0 streams this CTA's weight tiles
//     of all stages through a ring of 7-8 slots (free-running, HBM -> smem), warp 1 fetches the activation tile of each (item, chunk)
//     once its counter is complete, warp 2 issues tcgen05.mma (weights = A operand, M = 128; the chunk's rows = B operand,
//     N = CH; fp32 accumulator in a ring of TMEM column slots), warps 4-7 drain TMEM -> smem -> L2 with TMA reduce-add and
//     publish the chunk.  SIMT engine: warps 8-15 run the row-wise stages (bias / gate / residual / LayerNorm / AdaLN
//     modulate, band attention, GELU, CFG combine + ODE update) on the units of each (stage, chunk) dealt to this CTA.
//     The weight tiles of an item stay in shared memory while all chunks pass over them.  The row-wise units of a chunk run on
//     that chunk's own slice of the grid, so the in-order SIMT engine of a CTA serves one chain.
//   * The K slices of a tile meet in L2 through fp32 reduce-adds of partial sums rounded to a common quantum: exact, hence
//     order-independent sums - the same seed gives the same bits on every run (flow_quantize).
//
// What bounds a step (34 GEMM + row-wise stage pairs of ~9 us per evaluation) and every measured dead end: DESIGN.md section 6.
//
// Reference semantics: FMT.py:151-198 (block / decoder), :277-340 (forward), :342-401 (CFG), torchdiffeq fixed-grid solvers.
#pragma once
#include "window.cuh"

namespace fmt {

constexpr int FLOW_THREADS = 512;                // warps 0-2: W producer, A loader, MMA issuer; 3: idle; 4-7: epilogue; 8-15: SIMT
constexpr int FLOW_SIMT = 256;
constexpr int FLOW_SIMT_WARP0 = 8;
constexpr int FLOW_W_BYTES = 128 * 64 * 2;       // one weight tile: 128 features x 64 K, bf16
constexpr int FLOW_STG_BYTES = 32 * 128 * 4;     // epilogue staging: 32 rows x 128 features fp32
constexpr int FLOW_MAX_NW = 8, FLOW_MAX_NA = 4, FLOW_MAX_TS = 16;
constexpr int FLOW_MAX_GEMMS = 2 + 4 * WIN_MAX_DEPTH;
constexpr int FLOW_MAX_CHUNKS = 32;
constexpr int FLOW_FLAG_STRIDE = 8;              // uints between two counters (one 32-byte sector each)
constexpr int FLOW_BAR_BYTES = 1024;
constexpr int FLOW_SMEM_MAX = 222 * 1024;        // dynamic shared memory the host may hand out (rings + staging + barriers)

struct FlowGemm {
  int tm_w, tm_acc;          // tensor maps: weights (box 64 K x 128 features), accumulator (box 128 features x 32 rows, fp32)
  int n_ft, nkb, pk;         // feature tiles, K blocks, K splits; item i = (ft = i % n_ft, ks = i / n_ft) runs on CTA (i + cta_off) % grid
  int cta_off;
  int a_src;                 // 0: row-major ODE-state operand `ax` through tensor map tm_ax; 1: A1, 2: A2, 3: Hm (pre-tiled, bulk copies)
  int n_items;
  int par_blk;               // qkv GEMM of block par_blk: accumulates into QKV buffer (evaluation * depth + block) & 1 = map tm_acc + parity; else -1
};

struct FlowParams {
  ModelShape s;
  int R, depth, heads, window, mlp_hidden, NT;
  int n_steps, n_stages, n_gemms;
  int CH, nsub, NPs, n_chunks, RP;     // rows per chunk, chunks per sequence, padded rows per sequence, chunks, padded rows in total
  int nw, na, a_slot_bytes, n_tslots;  // weight ring slots, activation ring slots and their size, TMEM column slots (512 / CH)
  int tm_ax, poll_mode;
  float fx_c;                          // deterministic split-K: partial sums are rounded to multiples of 2^-k with (v + fx_c) - fx_c; 0 = off
  const FlowGemm* gemms;               // device array [n_gemms]: x_emb, (qkv, proj, fc1, fc2) x depth, dec
  const CUtensorMap* tmaps;
  float *X, *Pacc, *QKVacc, *Hacc, *Vacc;          // padded rows; QKVacc holds two buffers (block parity)
  __nv_bfloat16 *A1, *A2, *Hm, *ax;                // A1 / A2 / Hm: [chunk][K block][CH][64] bf16, 128-byte swizzle applied
  const __nv_bfloat16* table;                      // (n_eval, U, NT): one row per DISTINCT condition row
  const int* urow;                                 // table row of every token row (nullptr: identity, U = R)
  int U;
  const float *b_x, *pos, *b_dec;
  const float *b_qkv[WIN_MAX_DEPTH], *b_proj[WIN_MAX_DEPTH], *b_fc1[WIN_MAX_DEPTH], *b_fc2[WIN_MAX_DEPTH];
  float *x_state, *kbuf;
  const float* ddt;
  float rk_a[16], rk_b[4];
  const WindowArgs* wargs;
  unsigned *g_done, *s_done;           // [n_eval][n_gemms][n_chunks] counters, FLOW_FLAG_STRIDE apart, zeroed before every launch
  int* err_flag;
  long long* trace;                    // optional (FMT_WIN_TRACE=1): [cta][2][n_gemms][n_chunks][8] SM-clock stamps, then [cta][2][2] calibration pairs of evaluation trace_eval
  int trace_eval;
  long long spin_limit;
};

// per-CTA copy of what the role warps need about each GEMM instance (shared memory: 32 bytes per instance)
struct FlowItem { int ft, kb0, kb1, tm_w, tm_acc, a_src, n_items, nkb, par_blk, pad0, pad1, pad2; };   // par_blk >= 0: qkv of that block (accumulator map + parity)
// per chunk: sequence, first frame, valid rows, first real row (table / ax / pos index), first padded row
struct FlowChunk { int seq, f0, vr, rr0, rp0, sub, clip, pad; };
// per (SIMT kind, chunk): first unit of this CTA (-1: none), number of units, participating CTAs, unit stride of a CTA
struct FlowUnits { int u0, n_units, n_part, stride, pad; };
enum { FK_ROW = 0, FK_ATTN = 1, FK_GELU = 2, FK_COMB = 3 };

struct FlowSmem {
  uint8_t *wring, *aring;
  float* stg;
  uint64_t *w_full, *w_empty, *a_full, *a_empty, *t_full, *t_empty;
  uint32_t* tmem_slot;
};

// Operand layout: element (row r of chunk c, column col) of an activation with nkb K blocks
__device__ __forceinline__ size_t flow_tiled_off(int c, int r, int col, int nkb, int CH) {
  const int kb = col >> 6, cc = col & 63;
  return (static_cast<size_t>(c) * nkb + kb) * (CH * 64) + static_cast<size_t>(r) * 64 + ((((cc >> 3) ^ (r & 7)) << 3) | (cc & 7));
}

__device__ __forceinline__ void flow_fail(const FlowParams& p, int code) { win_fail(p.err_flag, code); }

// Deterministic split-K.  The K slices of a tile meet in L2 through fp32 reduce-adds in arrival order.  Every partial sum is first
// rounded to a multiple of the quantum q = 2^-FMT_FLOW_FIXED (two FADDs: (v + C) - C with C = 1.5 * 2^23 * q); sums of multiples of q
// are exact in fp32 while they stay below 2^24 * q, exact additions are associative, and so the same inputs give the same bits on
// every run (the reference is bitwise reproducible under fix_noise_seed, nodes_vadv.py:673-689).  q = 2^-14: exact below 1024, each
// partial moves by at most 3.1e-5 (bf16 rounding of the operands moves a value of 1 by 2e-3).  Beyond the range the additions round
// as usual: the result stays fp32-accurate and merely loses run-to-run bit equality.
__device__ __forceinline__ float flow_quantize(const FlowParams& p, float v) { return __fsub_rn(__fadd_rn(v, p.fx_c), p.fx_c); }

__device__ __forceinline__ void flow_mbar_wait(const FlowParams& p, uint64_t* bar, uint32_t parity, int code) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > p.spin_limit) flow_fail(p, code);
  }
}
// spin until the counter has reached `target` (acquire)
__device__ __forceinline__ unsigned ld_relaxed_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// poll_mode 1: relaxed polls (no L1 invalidation per poll - the other engine of the CTA keeps its L1 lines while this one waits) and
// one acquire load once the counter is complete; poll_mode 0: every poll is an acquire load
__device__ __forceinline__ int flow_wait_flag(const FlowParams& p, const unsigned* flag, unsigned target, int code) {
  if (target == 0u) return 0;
  if (ld_acquire_gpu(flag) >= target) return 1;
  const long long t0 = clock64();
  int polls = 2;
  if (p.poll_mode == 1) {
    while (ld_relaxed_gpu(flag) < target) {
      ++polls;
      if (clock64() - t0 > p.spin_limit) flow_fail(p, code);
    }
    (void)ld_acquire_gpu(flag);
  } else {
    while (ld_acquire_gpu(flag) < target) {
      ++polls;
      if (clock64() - t0 > p.spin_limit) flow_fail(p, code);
    }
  }
  return polls;                                  // trace only
}
__device__ __forceinline__ unsigned* flow_flag(unsigned* base, const FlowParams& p, int e, int st, int c) {
  return base + (static_cast<size_t>(e) * p.n_gemms + st) * (static_cast<size_t>(p.n_chunks) * FLOW_FLAG_STRIDE) + c * FLOW_FLAG_STRIDE;
}
__device__ __forceinline__ void flow_mark(const FlowParams& p, int e, int eng, int st, int c, int slot) {
  if (p.trace != nullptr && e == p.trace_eval)
    p.trace[(((static_cast<size_t>(blockIdx.x) * 2 + eng) * p.n_gemms + st) * p.n_chunks + c) * 8 + slot] = clock64();
}
// SM clocks of different SMs are unrelated: every CTA stamps its clock right after a grid-wide rendezvous at kernel start and end
// (skew = one L2 round trip), and the global timer beside it; the trace tool maps every stamp to a common time base with them
__device__ __forceinline__ void flow_calibrate(const FlowParams& p, int which) {
  unsigned* ctr = p.s_done + static_cast<size_t>(p.n_steps * p.n_stages) * p.n_gemms * p.n_chunks * FLOW_FLAG_STRIDE + which * FLOW_FLAG_STRIDE;
  red_release_gpu_add(ctr, 1u);
  while (ld_acquire_gpu(ctr) < gridDim.x) {}
  const long long c = clock64();
  unsigned long long g;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
  long long* cal = p.trace + static_cast<size_t>(gridDim.x) * 2 * p.n_gemms * p.n_chunks * 8 + (static_cast<size_t>(blockIdx.x) * 2 + which) * 2;
  cal[0] = static_cast<long long>(g); cal[1] = c;
}
__device__ __forceinline__ int flow_simt_kind(const FlowParams& p, int si) {
  if (si == 0) return FK_ROW;
  if (si == p.n_gemms - 1) return FK_COMB;
  const int j = (si - 1) & 3;
  return j == 0 ? FK_ATTN : j == 2 ? FK_GELU : FK_ROW;
}

// ------------------------------------------------------------------------------------------------------ GEMM engine
// warp 0: weight tiles of this CTA's items, in stage order, as far ahead as the ring allows
__device__ __forceinline__ void flow_weight_producer(const FlowParams& p, const FlowItem* items, const FlowSmem& sm, int n_eval) {
  int slot = 0; uint32_t phase = 0;
  for (int e = 0; e < n_eval; ++e) {
    for (int g = 0; g < p.n_gemms; ++g) {
      const FlowItem it = items[g];
      if (it.ft < 0) continue;
      for (int kb = it.kb0; kb < it.kb1; ++kb) {
        flow_mbar_wait(p, &sm.w_empty[slot], phase ^ 1, 0x01000000 | (e << 16) | (g << 8));
        mbar_expect_tx(&sm.w_full[slot], FLOW_W_BYTES);
        tma_load_2d(&p.tmaps[it.tm_w], &sm.w_full[slot], sm.wring + slot * FLOW_W_BYTES, kb * 64, it.ft * 128, kEvictFirst);
        if (++slot == p.nw) { slot = 0; phase ^= 1; }
      }
    }
  }
}

// warp 1: the activation tile [CH rows x (kb1 - kb0) K blocks] of every (item, chunk), requested the moment the stage that writes
// it has finished the chunk
__device__ __forceinline__ void flow_act_loader(const FlowParams& p, const FlowItem* items, const FlowChunk* chunks, const FlowUnits* units,
                                                const FlowSmem& sm, int n_eval) {
  int slot = 0; uint32_t phase = 0;
  const int nc = p.n_chunks, CH = p.CH;
  for (int e = 0; e < n_eval; ++e) {
    for (int g = 0; g < p.n_gemms; ++g) {
      const FlowItem it = items[g];
      if (it.ft < 0) continue;
      const int nk = it.kb1 - it.kb0;
      const uint32_t bytes = static_cast<uint32_t>(nk) * CH * 128;
      const int kind = g == 0 ? FK_COMB : flow_simt_kind(p, g - 1);
      for (int c = 0; c < nc; ++c) {
        flow_mark(p, e, 0, g, c, 0);
        // dependency: the SIMT stage that produced this chunk of the operand (x-embedder: the CFG combine of the previous evaluation)
        if (g > 0) {
          const int polls = flow_wait_flag(p, flow_flag(p.s_done, p, e, g - 1, c), units[kind * FLOW_MAX_CHUNKS + c].n_part, 0x02000000 | (e << 16) | (g << 8) | c);
          if (p.trace != nullptr && e == p.trace_eval)
            p.trace[(((static_cast<size_t>(blockIdx.x) * 2) * p.n_gemms + g) * p.n_chunks + c) * 8 + 6] = polls;
        } else if (e > 0) {
          const int cc = chunks[c].clip * p.nsub + chunks[c].sub;          // the combine publishes per (clip, sub-chunk) on branch 0's chunk
          flow_wait_flag(p, flow_flag(p.s_done, p, e - 1, p.n_gemms - 1, cc), units[FK_COMB * FLOW_MAX_CHUNKS + cc].n_part,
                         0x02000000 | (e << 16) | (g << 8) | c);
        }
        fence_proxy_async_all();                                            // acquired generic-proxy writes -> this thread's async-proxy reads
        flow_mark(p, e, 0, g, c, 1);
        flow_mbar_wait(p, &sm.a_empty[slot], phase ^ 1, 0x03000000 | (e << 16) | (g << 8) | c);
        flow_mark(p, e, 0, g, c, 2);
        mbar_expect_tx(&sm.a_full[slot], bytes);
        uint8_t* dst = sm.aring + slot * p.a_slot_bytes;
        if (it.a_src == 0) {
          for (int j = 0; j < nk; ++j)
            tma_load_2d(&p.tmaps[p.tm_ax], &sm.a_full[slot], dst + j * CH * 128, (it.kb0 + j) * 64, chunks[c].rr0, kEvictLast);
        } else {
          const __nv_bfloat16* base = it.a_src == 1 ? p.A1 : it.a_src == 2 ? p.A2 : p.Hm;
          bulk_load_1d(dst, base + (static_cast<size_t>(c) * it.nkb + it.kb0) * (CH * 64), bytes, &sm.a_full[slot]);
        }
        if (++slot == p.na) { slot = 0; phase ^= 1; }
      }
    }
  }
}

// warp 2: D[128 features x CH rows] (+)= W[128 x 16] . A[CH x 16]^T, chunk after chunk over the resident weight tiles of the item
__device__ __forceinline__ void flow_mma_issuer(const FlowParams& p, const FlowItem* items, const FlowSmem& sm, uint32_t tmem_base, int n_eval) {
  const int nc = p.n_chunks, CH = p.CH;
  const uint32_t idesc = make_idesc_bf16_f32(128, static_cast<uint32_t>(CH));
  const uint64_t desc_hi = make_sw128_kmajor_desc(0);
  const uint32_t w_base = smem_u32(sm.wring) >> 4, a_base = smem_u32(sm.aring) >> 4;
  const uint32_t a_slot16 = static_cast<uint32_t>(p.a_slot_bytes) >> 4, a_kb16 = static_cast<uint32_t>(CH * 128) >> 4;
  const bool leader = elect_one();
  int w_slot = 0, a_slot = 0, t_slot = 0;
  uint32_t w_phase = 0, a_phase = 0, t_phase = 0;
  for (int e = 0; e < n_eval; ++e) {
    for (int g = 0; g < p.n_gemms; ++g) {
      const FlowItem it = items[g];
      if (it.ft < 0) continue;
      const int nk = it.kb1 - it.kb0;
      for (int c = 0; c < nc; ++c) {
        flow_mbar_wait(p, &sm.t_empty[t_slot], t_phase ^ 1, 0x04000000 | (e << 16) | (g << 8) | c);
        flow_mbar_wait(p, &sm.a_full[a_slot], a_phase, 0x05000000 | (e << 16) | (g << 8) | c);
        if (leader) flow_mark(p, e, 0, g, c, 7);                         // trace: the activation tile has landed
        int ws = w_slot; uint32_t wp = w_phase;
        const uint32_t d_addr = tmem_base + static_cast<uint32_t>(t_slot * CH);
        const bool last_chunk = c == nc - 1;
        for (int j = 0; j < nk; ++j) {
          if (c == 0) flow_mbar_wait(p, &sm.w_full[ws], wp, 0x06000000 | (e << 16) | (g << 8) | j);
          tc_fence_after();
          if (leader) {
            const uint64_t dw = desc_hi | (w_base + ws * (FLOW_W_BYTES >> 4)), da = desc_hi | (a_base + a_slot * a_slot16 + j * a_kb16);
            umma_bf16(d_addr, dw, da, idesc, j > 0 ? 1u : 0u);
            umma_bf16(d_addr, dw + 2, da + 2, idesc, 1u);
            umma_bf16(d_addr, dw + 4, da + 4, idesc, 1u);
            umma_bf16(d_addr, dw + 6, da + 6, idesc, 1u);
            if (last_chunk) umma_commit(&sm.w_empty[ws]);                  // every chunk has passed over this weight tile
          }
          if (++ws == p.nw) { ws = 0; wp ^= 1; }
        }
        if (leader) {
          umma_commit(&sm.a_empty[a_slot]);
          umma_commit(&sm.t_full[t_slot]);
        }
        __syncwarp();
        if (last_chunk) { w_slot = ws; w_phase = wp; }
        if (++a_slot == p.na) { a_slot = 0; a_phase ^= 1; }
        if (++t_slot == p.n_tslots) { t_slot = 0; t_phase ^= 1; }
      }
    }
  }
}

// warps 4-7: TMEM (lanes = features, columns = the chunk's rows) -> smem [row][feature] -> L2 reduce-add, then publish the chunk.
// The flag of a chunk is published once its reduce-adds have COMPLETED; when the next accumulator is already waiting, its tile
// is staged and sent first (the completion of the previous one is awaited behind it), so the TMA path never idles.
__device__ __forceinline__ void flow_epilogue(const FlowParams& p, const FlowItem* items, const FlowChunk* chunks, const FlowSmem& sm,
                                              uint32_t tmem_base, int n_eval) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int quarter = warp & 3, fl = quarter * 32 + lane;
  const bool issuer = (warp == 4 && lane == 0);
  const int nc = p.n_chunks, CH = p.CH, nh = CH >> 5;
  int t_slot = 0; uint32_t t_phase = 0;
  int stg_i = 0, n_sent = 0;
  unsigned* pending = nullptr;                      // issuer only: flag of the chunk whose reduce-adds are still in flight
  int pend_e = 0, pend_g = 0, pend_c = 0;
  for (int e = 0; e < n_eval; ++e) {
    for (int g = 0; g < p.n_gemms; ++g) {
      const FlowItem it = items[g];
      if (it.ft < 0) continue;
      const int tm_acc = it.tm_acc + (it.par_blk >= 0 ? ((e * p.depth + it.par_blk) & 1) : 0);
      for (int c = 0; c < nc; ++c) {
        if (lane == 0) flow_mbar_wait(p, &sm.t_full[t_slot], t_phase, 0x07000000 | (e << 16) | (g << 8) | c);
        __syncwarp();
        tc_fence_after();
        if (issuer) flow_mark(p, e, 0, g, c, 3);
        for (int h = 0; h < nh; ++h) {
          float* stg = sm.stg + stg_i * (FLOW_STG_BYTES / 4);
          float v[32];
          tmem_ld32(tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(t_slot * CH + h * 32), v);
          if (n_sent >= 2) {                        // the reduce that read this staging buffer two tiles ago must be done reading it
            if (issuer) bulk_wait_read<1>();
            named_bar_sync(2, 128);
          }
          tmem_ld_wait();
          if (p.fx_c != 0.f) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = flow_quantize(p, v[j]);
          }
          if (h == nh - 1) {                        // accumulator slot drained: hand it back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.t_empty[t_slot]);
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) stg[j * 128 + fl] = v[j];
          fence_proxy_async();                      // smem writes -> visible to the async proxy
          named_bar_sync(2, 128);
          if (issuer) {
            tma_reduce_add_2d(&p.tmaps[tm_acc], stg, it.ft * 128, chunks[c].rp0 + h * 32);
            bulk_commit();
          }
          stg_i ^= 1; ++n_sent;
        }
        if (issuer) {
          flow_mark(p, e, 0, g, c, 4);
          if (pending != nullptr) {                 // the previous chunk: everything but this chunk's nh groups has completed
            if (nh == 1) bulk_wait<1>(); else bulk_wait<2>();
            fence_proxy_async_all();
            red_release_gpu_add(pending, 1u);
            flow_mark(p, pend_e, 0, pend_g, pend_c, 5);
            pending = nullptr;
          }
          // is the next accumulator already there?  then keep the TMA path busy and publish this chunk behind it
          int nt = t_slot + 1; uint32_t nph = t_phase;
          if (nt == p.n_tslots) { nt = 0; nph ^= 1; }
          unsigned* flag = flow_flag(p.g_done, p, e, g, c);
          if (mbar_try_wait(&sm.t_full[nt], nph)) {
            pending = flag; pend_e = e; pend_g = g; pend_c = c;
          } else {
            bulk_wait<0>();
            fence_proxy_async_all();
            red_release_gpu_add(flag, 1u);
            flow_mark(p, e, 0, g, c, 5);
          }
        }
        if (++t_slot == p.n_tslots) { t_slot = 0; t_phase ^= 1; }
      }
    }
  }
  if (issuer && pending != nullptr) {
    bulk_wait<0>();
    fence_proxy_async_all();
    red_release_gpu_add(pending, 1u);
  }
  if (issuer) bulk_wait<0>();
}

// ------------------------------------------------------------------------------------------------------ SIMT engine
// thread index inside the SIMT engine: 0..255; warp index 0..7
__device__ __forceinline__ int flow_stid() { return static_cast<int>(threadIdx.x) - FLOW_SIMT_WARP0 * 32; }

// The dependency of one (stage, chunk): up to 4 counters that must reach `need`.  Every unit function issues the loads that do
// NOT depend on the GEMM (AdaLN table rows from HBM, residual, biases) first and only then calls flow_simt_wait, so that their
// latency hides behind the wait.
struct FlowWait {
  const unsigned* f0;      // counter of the chunk itself
  int stride1, stride2, n; // counter i >= 1 of n sits at f0 + stride1 + (i - 1) * stride2  (no pointer array: no local memory)
  unsigned need;
  int code;
  int e, si, c;
};
__device__ __forceinline__ void flow_simt_wait(const FlowParams& p, const FlowWait& w) {
  if (flow_stid() == 0) {
    flow_wait_flag(p, w.f0, w.need, w.code);
    if (w.n > 1) flow_wait_flag(p, w.f0 + w.stride1, w.need, w.code);
    for (int i = 2; i < w.n; ++i) flow_wait_flag(p, w.f0 + w.stride1 + (i - 1) * w.stride2, w.need, w.code);
    flow_mark(p, w.e, 1, w.si, w.c, 1);
  }
  named_bar_sync(1, FLOW_SIMT);
}

// ROW units: RPU token rows per unit, WPR warps per row (FPL float4 per lane each).
//   mode 0 (after x_embedder): X = acc + bias + pos_embed[frame]                       (FMT.py:319-320)
//   mode 1 (after proj / fc2): X = X + gate * (acc + bias)                             (FMT.py:174-175)
// then A1 = bf16( LayerNorm(X) * (1 + scale) + shift ) with this evaluation's table row (FMT.py:168-169,174-175,197); the
// accumulator row is zeroed for its next use.
template <int NV>
__device__ __forceinline__ void flow_row_units(const FlowParams& p, const FlowChunk& ck, int c, const FlowUnits& un, float* red_smem,
                                               const __nv_bfloat16* __restrict__ table_e, int mode, const float* __restrict__ bias, long long gate_off,
                                               long long shift_off, long long scale_off, const FlowWait& w) {
  constexpr int WPR = NV >= 4 ? 4 : NV;          // warps per row
  constexpr int FPL = NV / WPR;                  // float4 per lane
  constexpr int RPU = 8 / WPR;                   // rows per unit
  const int lane = threadIdx.x & 31, mw = (threadIdx.x >> 5) - FLOW_SIMT_WARP0;
  const int rsub = mw / WPR, wr = mw % WPR;
  const int H = p.s.H;
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  const int c0 = wr * (FPL * 128) + lane * 4;
  bool waited = false;
  for (int u = un.u0; u < un.n_units; u += un.stride) {
    const int r = u * RPU + rsub;
    const bool valid = r < ck.vr;
    const size_t prow = static_cast<size_t>(ck.rp0 + (valid ? r : 0));
    float* acc = p.Pacc + prow * H + c0;
    float* xr = p.X + prow * H + c0;
    const int trow_i = ck.rr0 + (valid ? r : 0);
    const __nv_bfloat16* trow = table_e + static_cast<size_t>(p.urow != nullptr ? __ldg(p.urow + trow_i) : trow_i) * p.NT + c0;
    float4 a[FPL], x[FPL], b[FPL], ps[FPL];
    uint2 tg[FPL], tsh[FPL], tsc[FPL];
    // unconditional (row 0 stands in for a row past the chunk): conditionally defined registers would be demoted to local memory
#pragma unroll
    for (int i = 0; i < FPL; ++i) {
      tsh[i] = ld_nc_u2(trow + shift_off + i * 128);
      tsc[i] = ld_nc_u2(trow + scale_off + i * 128);
      b[i] = __ldg(reinterpret_cast<const float4*>(bias + c0 + i * 128));
      if (mode == 1) {
        x[i] = ldcg4(xr + i * 128);
        tg[i] = ld_nc_u2(trow + gate_off + i * 128);
      } else {
        ps[i] = __ldg(reinterpret_cast<const float4*>(p.pos + static_cast<size_t>(ck.f0 + (valid ? r : 0)) * H + c0 + i * 128));
      }
    }
    if (!waited) { flow_simt_wait(p, w); waited = true; }
    if (!valid) continue;
#pragma unroll
    for (int i = 0; i < FPL; ++i) a[i] = ldcg4(acc + i * 128);
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < FPL; ++i) {
      if (mode == 0) {
        x[i] = make_float4(a[i].x + b[i].x + ps[i].x, a[i].y + b[i].y + ps[i].y, a[i].z + b[i].z + ps[i].z, a[i].w + b[i].w + ps[i].w);
      } else {
        float g[4];
        bf16x4_to_f32(tg[i], g);
        x[i].x = fmaf(g[0], a[i].x + b[i].x, x[i].x); x[i].y = fmaf(g[1], a[i].y + b[i].y, x[i].y);
        x[i].z = fmaf(g[2], a[i].z + b[i].z, x[i].z); x[i].w = fmaf(g[3], a[i].w + b[i].w, x[i].w);
      }
      sum += (x[i].x + x[i].y) + (x[i].z + x[i].w);
    }
#pragma unroll
    for (int i = 0; i < FPL; ++i) {
      *reinterpret_cast<float4*>(xr + i * 128) = x[i];
      *reinterpret_cast<float4*>(acc + i * 128) = zero4;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    float* red = red_smem + rsub * 16;
    if (WPR > 1) {
      if (lane == 0) red[wr] = sum;
      named_bar_sync(3 + rsub, WPR * 32);
      sum = 0.f;
#pragma unroll
      for (int k = 0; k < WPR; ++k) sum += red[k];
    }
    const float mean = sum / static_cast<float>(H);
    float var = 0.f;
#pragma unroll
    for (int i = 0; i < FPL; ++i) {
      const float d0 = x[i].x - mean, d1 = x[i].y - mean, d2 = x[i].z - mean, d3 = x[i].w - mean;
      var += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) var += __shfl_xor_sync(0xffffffffu, var, o);
    if (WPR > 1) {
      if (lane == 0) red[8 + wr] = var;
      named_bar_sync(3 + rsub, WPR * 32);
      var = 0.f;
#pragma unroll
      for (int k = 0; k < WPR; ++k) var += red[8 + k];
    }
    const float rstd = rsqrtf(var / static_cast<float>(H) + 1e-6f);
    const int nkb = H >> 6;
#pragma unroll
    for (int i = 0; i < FPL; ++i) {
      float sh[4], sc[4];
      bf16x4_to_f32(tsh[i], sh);
      bf16x4_to_f32(tsc[i], sc);
      float v[4] = {(x[i].x - mean) * rstd, (x[i].y - mean) * rstd, (x[i].z - mean) * rstd, (x[i].w - mean) * rstd};
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] = fmaf(v[k], 1.f + sc[k], sh[k]);
      *reinterpret_cast<uint2*>(p.A1 + flow_tiled_off(c, r, c0 + i * 128, nkb, p.CH)) = f32x4_to_bf16(v);
    }
    if (WPR > 1) named_bar_sync(3 + rsub, WPR * 32);      // `red` is reused by the next row
  }
  if (!waited) flow_simt_wait(p, w);
}

// ATTN units: a unit = (one head, one group of consecutive row pairs of the chunk); inside it a warp takes a row pair, one row per
// half warp, DPL = head_dim / 16 dimensions per lane: band-masked attention (FMT.py:15-19,69-88) straight from the fp32 QKV
// accumulator of this block's parity (+ qkv bias).
//   * A CTA's L2 -> SM path moves ~32 B per clock, so what a CTA fetches decides the stage: consecutive rows of ONE head share all
//     but a halo of their keys, and the q / k / v loads are ordinary cached loads - the acquire poll in front of them invalidated the
//     L1, the first warp to touch a line fetches it, the other warps of the CTA hit (or merge with the miss).  A unit of 10 rows reads
//     (10 + 14 + 14) x 512 B instead of 10 x 11 x 512 B.
//   * Everything after the loads is a dependent chain executed by ONE warp, so it is laid out for few instructions: dot products
//     reduce over 16 lanes (4 shuffle rounds serve both rows), the softmax over a batch of keys is the plain two-pass form (max, then
//     independent exponentials) and batches are merged online only when the band is wider than KB keys.
// Keys / values of the neighbouring chunk of the same sequence are read across the chunk boundary.  Also zeroes the rows' slices in the
// OTHER parity buffer (read for the last time one block ago).
template <int VL> struct F32VecCa;
template <> struct F32VecCa<2> { static __device__ __forceinline__ void ld(const float* p, float (&v)[2]) { float2 t = *reinterpret_cast<const float2*>(p); v[0] = t.x; v[1] = t.y; } };
template <> struct F32VecCa<4> { static __device__ __forceinline__ void ld(const float* p, float (&v)[4]) { float4 t = *reinterpret_cast<const float4*>(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; } };
template <int DPL>
__device__ __forceinline__ void flow_attn_units(const FlowParams& p, const FlowChunk& ck, int c, const FlowUnits& un, const float* __restrict__ qkv,
                                                float* __restrict__ qkv_other, const float* __restrict__ bqkv, const FlowWait& w) {
  const int lane = threadIdx.x & 31, mw = (threadIdx.x >> 5) - FLOW_SIMT_WARP0;
  constexpr int hd = DPL * 16;
  constexpr int VL = DPL >= 4 ? 4 : DPL, NVL = DPL / VL;        // vector loads of VL floats, NVL per row
  const int half = lane >> 4, sl = lane & 15;
  const int N = p.s.N, heads = p.heads, H = p.s.H, ld = 3 * H, win = p.window;
  const float scale = rsqrtf(static_cast<float>(hd));
  const size_t seq_row0 = static_cast<size_t>(ck.seq) * p.NPs;
  const int n_rp = (ck.vr + 1) >> 1;                             // row pairs of the chunk
  const int n_grp = un.n_units / heads;                          // groups of row pairs per head
  const int ppg = (n_rp + n_grp - 1) / n_grp;                    // row pairs per group
  // the biases of the first unit's head do not depend on the GEMM: fetched before the wait (the poll invalidates the L1 under them)
  float bqv[DPL], bk[DPL], bv[DPL];
  int hb = (un.u0 >= 0 ? un.u0 : 0) % heads;
#pragma unroll
  for (int k = 0; k < DPL; ++k) {
    const float* bq = bqkv + hb * hd + sl * DPL;
    bqv[k] = __ldg(bq + k); bk[k] = __ldg(bq + H + k); bv[k] = __ldg(bq + 2 * H + k);
  }
  flow_simt_wait(p, w);
  for (int u = un.u0; u < un.n_units; u += un.stride)
  for (int pp = mw; pp < ppg; pp += 8) {
    const int g = u / heads, hh = u - g * heads;                 // one division per stage per warp (off the flag path)
    const int rp = g * ppg + pp;
    if (rp >= n_rp) continue;
    if (hh != hb) {                                              // a CTA with several units (more chunks than CTAs per head): reload
      hb = hh;
#pragma unroll
      for (int k = 0; k < DPL; ++k) {
        const float* bq = bqkv + hb * hd + sl * DPL;
        bqv[k] = __ldg(bq + k); bk[k] = __ldg(bq + H + k); bv[k] = __ldg(bq + 2 * H + k);
      }
    }
    const bool valid = 2 * rp + half < ck.vr;
    const int r = valid ? 2 * rp + half : 2 * rp;              // an odd last row: the upper half warp shadows the lower one and stores nothing
    const int fi = ck.f0 + r;
    const float* base = qkv + seq_row0 * ld + hh * hd + sl * DPL;
    const int j0 = max(0, fi - win), j1 = min(N - 1, fi + win);
    const int n_keys = max(j1 - j0, __shfl_xor_sync(0xffffffffu, j1 - j0, 16)) + 1;    // warp-uniform trip count
    float q[DPL], acc[DPL];
#pragma unroll
    for (int i = 0; i < NVL; ++i) F32VecCa<VL>::ld(base + static_cast<size_t>(fi) * ld + i * VL, *reinterpret_cast<float(*)[VL]>(&q[i * VL]));
    float mx = -INFINITY, den = 0.f;
#pragma unroll
    for (int k = 0; k < DPL; ++k) acc[k] = 0.f;
    constexpr int KB = 5;
    bool first = true;
#pragma unroll 1
    for (int jb = 0; jb < n_keys; jb += KB) {
      float kv[KB][DPL], vv[KB][DPL], sc[KB];
#pragma unroll
      for (int t = 0; t < KB; ++t) {
        const int j = min(j0 + jb + t, j1);
#pragma unroll
        for (int i = 0; i < NVL; ++i) {
          F32VecCa<VL>::ld(base + static_cast<size_t>(j) * ld + H + i * VL, *reinterpret_cast<float(*)[VL]>(&kv[t][i * VL]));
          F32VecCa<VL>::ld(base + static_cast<size_t>(j) * ld + 2 * H + i * VL, *reinterpret_cast<float(*)[VL]>(&vv[t][i * VL]));
        }
      }
      if (first) {
#pragma unroll
        for (int k = 0; k < DPL; ++k) q[k] = (q[k] + bqv[k]) * scale;
        first = false;
      }
#pragma unroll
      for (int t = 0; t < KB; ++t) {
        float d = 0.f;
#pragma unroll
        for (int k = 0; k < DPL; ++k) d = fmaf(q[k], kv[t][k] + bk[k], d);
        sc[t] = d;
      }
      if (flow_stid() == 0) flow_mark(p, w.e, 1, w.si, w.c, 5);
#pragma unroll
      for (int o = 8; o > 0; o >>= 1)
#pragma unroll
        for (int t = 0; t < KB; ++t) sc[t] += __shfl_xor_sync(0xffffffffu, sc[t], o);
      if (flow_stid() == 0) flow_mark(p, w.e, 1, w.si, w.c, 6);
      float bm = -INFINITY;
#pragma unroll
      for (int t = 0; t < KB; ++t) {
        if (j0 + jb + t > j1) sc[t] = -INFINITY;
        bm = fmaxf(bm, sc[t]);
      }
      const float nmx = fmaxf(mx, bm);                           // finite: the first batch of a row always holds a valid key
      const float corr = __expf(mx - nmx);
      float ps = 0.f, pr[KB];
#pragma unroll
      for (int t = 0; t < KB; ++t) { pr[t] = __expf(sc[t] - nmx); ps += pr[t]; }
      den = fmaf(den, corr, ps);
#pragma unroll
      for (int k = 0; k < DPL; ++k) {
        float a = acc[k] * corr;
#pragma unroll
        for (int t = 0; t < KB; ++t) a = fmaf(pr[t], vv[t][k], a);
        acc[k] = a;
      }
      mx = nmx;
    }
    if (flow_stid() == 0) flow_mark(p, w.e, 1, w.si, w.c, 7);
    const float inv = __fdividef(1.f, den);
    float o[DPL];
#pragma unroll
    for (int k = 0; k < DPL; ++k) o[k] = fmaf(acc[k], inv, bv[k]);   // sum_c p_c (v_c + b) / den = sum_c p_c v_c / den + b
    if (valid) {
      // DPL <= 8 elements stay inside one 16-byte chunk of the swizzled operand tile
      __nv_bfloat16* op = p.A2 + flow_tiled_off(c, r, hh * hd + sl * DPL, H >> 6, p.CH);
      // q / k / v slices of (row, head) in the other parity buffer: every reader (this chunk's and the neighbours' previous ATTN
      // stage) finished before this block's qkv GEMM could complete
      float* z = qkv_other + (seq_row0 + fi) * ld + hh * hd + sl * DPL;
      if constexpr (DPL == 8) {
        uint4 t;
        const uint2 lo = f32x4_to_bf16(*reinterpret_cast<const float(*)[4]>(&o[0])), hi = f32x4_to_bf16(*reinterpret_cast<const float(*)[4]>(&o[4]));
        t.x = lo.x; t.y = lo.y; t.z = hi.x; t.w = hi.y;
        *reinterpret_cast<uint4*>(op) = t;
      } else if constexpr (DPL == 4) {
        *reinterpret_cast<uint2*>(op) = f32x4_to_bf16(*reinterpret_cast<const float(*)[4]>(&o[0]));
      } else {
#pragma unroll
        for (int k = 0; k < DPL; ++k) op[k] = __float2bfloat16_rn(o[k]);
      }
      if constexpr (DPL >= 4) {
        const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < DPL / 4; ++i) {
          *reinterpret_cast<float4*>(z + i * 4) = zero4; *reinterpret_cast<float4*>(z + H + i * 4) = zero4; *reinterpret_cast<float4*>(z + 2 * H + i * 4) = zero4;
        }
      } else {
#pragma unroll
        for (int k = 0; k < DPL; ++k) { z[k] = 0.f; z[H + k] = 0.f; z[2 * H + k] = 0.f; }
      }
    }
  }
}

// GELU units: a unit = one slab of 256 float4 (one row x 1024 columns) of the chunk: Hm = bf16( GELU_tanh(Hacc + b_fc1) ), Hacc <- 0
// (timm Mlp: fc1 -> act, FMT.py:159-162).  A CTA issues the loads of up to NB of its slabs before the first dependent instruction.
__device__ __forceinline__ void flow_gelu_units(const FlowParams& p, const FlowChunk& ck, int c, const FlowUnits& un, const float* __restrict__ b1,
                                                const FlowWait& w) {
  const int M4 = p.mlp_hidden, nkb = M4 >> 6;
  const int n_q = (M4 / 4 + FLOW_SIMT - 1) / FLOW_SIMT;        // slabs per row
  float* hacc = p.Hacc + static_cast<size_t>(ck.rp0) * M4;
  constexpr int NB = 5;
  const int stid = flow_stid();
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  flow_simt_wait(p, w);
#pragma unroll 1
  for (int u = un.u0; u < un.n_units; u += NB * un.stride) {
    float4 a[NB], b[NB];
    // slab sl -> (row, first column of this thread); recomputed for the stores instead of being kept in registers
    auto locate = [&](int k, int& row, int& col) -> bool {
      const int sl = u + k * un.stride;
      row = sl / n_q;
      col = ((sl - row * n_q) * FLOW_SIMT + stid) * 4;
      return sl < un.n_units && col < M4;
    };
#pragma unroll
    for (int k = 0; k < NB; ++k) {                  // unconditional loads (a clamped address when the slab is out of range): conditionally
      int row, col;                                 // defined registers would be demoted to local memory
      if (!locate(k, row, col)) { row = 0; col = 0; }
      a[k] = ldcg4(hacc + static_cast<size_t>(row) * M4 + col);
      b[k] = __ldg(reinterpret_cast<const float4*>(b1 + col));
    }
#pragma unroll
    for (int k = 0; k < NB; ++k) {
      int row, col;
      if (locate(k, row, col)) {
        float v[4] = {gelu_tanh_fast(a[k].x + b[k].x), gelu_tanh_fast(a[k].y + b[k].y), gelu_tanh_fast(a[k].z + b[k].z), gelu_tanh_fast(a[k].w + b[k].w)};
        *reinterpret_cast<uint2*>(p.Hm + flow_tiled_off(c, row, col, nkb, p.CH)) = f32x4_to_bf16(v);
        *reinterpret_cast<float4*>(hacc + static_cast<size_t>(row) * M4 + col) = zero4;
      }
    }
  }
}

// COMB unit = 256 elements (frame, column) of the current frames of one (clip, sub-chunk): decoder bias, CFG combine
// (FMT.py:375-379,396-399), then the explicit Runge-Kutta bookkeeping of stage g of step `step` (Euler: y += dt * v).  Writes the
// x-embedder operand `ax` of the next evaluation (all branches) and zeroes Vacc.
__device__ __forceinline__ void flow_comb_unit(const FlowParams& p, const FlowChunk& ck, int unit, int step, int g) {
  const ModelShape& s = p.s;
  const int G = p.n_stages;
  const int fc0 = max(ck.f0, s.P);                                  // first current frame of the sub-chunk
  const int n_el = max(0, ck.f0 + ck.vr - fc0) * s.W;
  const int i = unit * FLOW_SIMT + flow_stid();
  if (i >= n_el) return;
  const int f = fc0 + i / s.W, j = i - (i / s.W) * s.W;
  const int b = ck.clip;
  const size_t nx = static_cast<size_t>(s.B) * s.L * s.W;
  const size_t o = (static_cast<size_t>(b) * s.L + (f - s.P)) * s.W + j;
  float vb[4];
  float* const va0 = p.Vacc + (static_cast<size_t>(b) * p.NPs + f) * s.W + j;          // branch br: + br * vstride
  const size_t vstride = static_cast<size_t>(s.B) * p.NPs * s.W;
#pragma unroll
  for (int br = 0; br < 4; ++br) vb[br] = __ldcg(va0 + (br < s.nb ? br : 0) * vstride);
  const float bd = __ldg(p.b_dec + j);
  const float dt = __ldg(p.ddt + step);
  const SlotArgs* const slots = p.wargs->slots;
  float a_s, r_s, e_s;
  int nb;
  const float y0 = __ldcg(p.x_state + o);
  float kprev[4] = {0.f, 0.f, 0.f, 0.f};
  if (G > 1) {
#pragma unroll
    for (int jj = 0; jj < 3; ++jj)
      if (jj < g) kprev[jj] = __ldcg(p.kbuf + static_cast<size_t>(jj) * nx + o);
  }
#pragma unroll
  for (int br = 0; br < 4; ++br)
    if (br < s.nb) { vb[br] += bd; va0[br * vstride] = 0.f; }
  slot_guidance(slots, s.nb, b, vb, nb, a_s, r_s, e_s);
  float v;
  if (nb == 1) v = vb[0];
  else if (nb == 3) v = vb[0] + a_s * (vb[2] - vb[0]) + e_s * (vb[1] - vb[2]);
  else v = vb[0] + r_s * (vb[1] - vb[0]) + a_s * (vb[3] - vb[1]) + e_s * (vb[2] - vb[3]);
  float y;
  if (G == 1) {
    y = fmaf(dt, v, y0);
    p.x_state[o] = y;
  } else {
    p.kbuf[static_cast<size_t>(g) * nx + o] = v;
    const bool last = (g == G - 1);
    const float* cf = last ? p.rk_b : &p.rk_a[(g + 1) * G];
    float acc = 0.f;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
      if (jj <= g && cf[jj] != 0.f) acc = fmaf(cf[jj], jj == g ? v : kprev[jj], acc);
    y = fmaf(dt, acc, y0);
    if (last) p.x_state[o] = y;
  }
  const __nv_bfloat16 t = __float2bfloat16_rn(y);
  for (int br = 0; br < s.nb; ++br) p.ax[((static_cast<size_t>(br) * s.B + b) * s.N + f) * s.W + j] = t;
}

template <int NV>
__device__ __forceinline__ void flow_simt_engine(const FlowParams& p, const FlowItem* items, const FlowChunk* chunks, const FlowUnits* units,
                                                 float* red_smem, int n_eval) {
  const int stid = flow_stid();
  const int nc = p.n_chunks, n_st = p.n_gemms, D = p.depth;
  const long long H = p.s.H;
  const size_t qkv_buf = static_cast<size_t>(p.RP) * 3 * H;
  const int hd = p.s.H / p.heads;
  for (int e = 0; e < n_eval; ++e) {
    const __nv_bfloat16* table_e = p.table + static_cast<size_t>(e) * (static_cast<size_t>(p.U) * p.NT);
    for (int si = 0; si < n_st; ++si) {
      const int kind = flow_simt_kind(p, si);
      const int blk = (si >= 1 && si < n_st - 1) ? (si - 1) >> 2 : 0;
      const int j = (si - 1) & 3;
      for (int c = 0; c < nc; ++c) {
        const FlowUnits un = units[kind * FLOW_MAX_CHUNKS + c];
        if (un.u0 < 0) continue;
        const FlowChunk ck = chunks[c];
        // ---- what this chunk's units read: every K slice x feature tile of the GEMM this stage consumes
        FlowWait w;
        w.need = static_cast<unsigned>(items[si].n_items);
        w.code = 0x08000000 | (e << 16) | (si << 8) | c;
        w.e = e; w.si = si; w.c = c; w.n = 1;
        w.f0 = flow_flag(p.g_done, p, e, si, c);
        w.stride1 = w.stride2 = 0;
        if (kind == FK_COMB) {                                              // the same (clip, sub-chunk) of every branch
          w.n = p.s.nb;
          w.stride1 = w.stride2 = p.s.B * p.nsub * FLOW_FLAG_STRIDE;
        } else if (kind == FK_ATTN) {                                       // the band crosses into the neighbouring chunks of the sequence
          const bool lo = ck.sub > 0, hi = ck.sub < p.nsub - 1;
          if (lo && hi) { w.n = 3; w.stride1 = -FLOW_FLAG_STRIDE; w.stride2 = 2 * FLOW_FLAG_STRIDE; }
          else if (lo) { w.n = 2; w.stride1 = -FLOW_FLAG_STRIDE; }
          else if (hi) { w.n = 2; w.stride1 = FLOW_FLAG_STRIDE; }
        }
        if (stid == 0) flow_mark(p, e, 1, si, c, 0);
        // ---- this CTA's units of (stage, chunk)
        if (kind == FK_ROW) {
          if (si == 0) {
            flow_row_units<NV>(p, ck, c, un, red_smem, table_e, 0, p.b_x, 0, 0, H, w);       // LN + modulate with block 0's (shift_msa, scale_msa)
          } else {
            const long long base = static_cast<long long>(blk) * 6 * H;
            const bool after_proj = (j == 1);
            const long long gate_off = base + (after_proj ? 2 : 5) * H;
            // after proj -> gate_msa, then the mlp modulation; after fc2 -> gate_mlp, then the NEXT block's msa modulation or,
            // after the last block, the decoder's (shift, scale)
            const long long mod = after_proj ? base + 3 * H : base + 6 * H;
            flow_row_units<NV>(p, ck, c, un, red_smem, table_e, 1, after_proj ? p.b_proj[blk] : p.b_fc2[blk], gate_off, mod, mod + H, w);
          }
        } else if (kind == FK_ATTN) {
          const int par = (e * D + blk) & 1;
          const float* q = p.QKVacc + par * qkv_buf;
          float* qo = p.QKVacc + (par ^ 1) * qkv_buf;
          if (hd == 128) flow_attn_units<8>(p, ck, c, un, q, qo, p.b_qkv[blk], w);
          else if (hd == 64) flow_attn_units<4>(p, ck, c, un, q, qo, p.b_qkv[blk], w);
          else flow_attn_units<2>(p, ck, c, un, q, qo, p.b_qkv[blk], w);
        } else if (kind == FK_GELU) {
          flow_gelu_units(p, ck, c, un, p.b_fc1[blk], w);
        } else {
          flow_simt_wait(p, w);
          for (int u = un.u0; u < un.n_units; u += un.stride) flow_comb_unit(p, ck, u, e / p.n_stages, e % p.n_stages);
        }
        // ---- publish: every thread's writes -> (proxy fence: they feed TMA reads / reduce-adds) -> one release
        if (stid == 0) flow_mark(p, e, 1, si, c, 2);
        fence_proxy_async_all();
        named_bar_sync(1, FLOW_SIMT);
        if (stid == 0) {
          flow_mark(p, e, 1, si, c, 3);
          red_release_gpu_add(flow_flag(p.s_done, p, e, si, c), 1u);
          flow_mark(p, e, 1, si, c, 4);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------- kernel
// The chunks and this CTA's units of every (SIMT kind, chunk), built by the CTA's FLOW_THREADS threads.  Units are dealt for a grid of
// at least n_chunks CTAs (the kernel runs one CTA per SM): with fewer, chunk c >= gridDim.x would get no CTA.
template <int NV>
__device__ __forceinline__ void flow_chunk_tables(const FlowParams& p, FlowChunk* chunks, FlowUnits* units, int nctas, int cta) {
  for (int c = threadIdx.x; c < p.n_chunks; c += FLOW_THREADS) {
    FlowChunk ck;
    ck.seq = c / p.nsub; ck.sub = c - ck.seq * p.nsub;
    ck.f0 = ck.sub * p.CH;
    ck.vr = min(p.CH, p.s.N - ck.f0);
    ck.rr0 = ck.seq * p.s.N + ck.f0;
    ck.rp0 = c * p.CH;
    ck.clip = ck.seq % p.s.B;
    ck.pad = 0;
    chunks[c] = ck;
    for (int kind = 0; kind < 4; ++kind) {
      int n_units;
      const int row_wpr = NV >= 4 ? 4 : NV;                                  // as in flow_row_units
      if (kind == FK_ROW) n_units = (ck.vr + 8 / row_wpr - 1) / (8 / row_wpr);
      else if (kind == FK_ATTN) n_units = p.heads * max(1, (nctas / p.n_chunks) / p.heads);   // (head, group of row pairs), see flow_attn_units
      else if (kind == FK_GELU) n_units = ck.vr * ((p.mlp_hidden / 4 + FLOW_SIMT - 1) / FLOW_SIMT);
      else n_units = ck.seq < p.s.B ? (max(0, ck.f0 + ck.vr - max(ck.f0, p.s.P)) * p.s.W + FLOW_SIMT - 1) / FLOW_SIMT : 0;   // published on branch 0's chunks
      // The row-wise stages of a chunk run on that chunk's own slice of the grid, so that the in-order SIMT engine of a CTA
      // serves ONE dependency chain and never holds a ready chunk back behind a late one; the CFG combine (once per
      // evaluation, needs every branch) is dealt over the whole grid.
      FlowUnits un;
      un.n_units = n_units; un.pad = 0;
      if (kind == FK_COMB) {
        const int rot = (c * 29) % nctas;
        int u0 = cta - rot;
        if (u0 < 0) u0 += nctas;
        un.stride = nctas; un.n_part = min(n_units, nctas); un.u0 = u0 < n_units ? u0 : -1;
      } else {
        const int gs = max(1, nctas / p.n_chunks);
        const int u0 = cta - c * gs;
        un.stride = gs; un.n_part = min(n_units, gs); un.u0 = (u0 >= 0 && u0 < gs && u0 < n_units) ? u0 : -1;
      }
      units[kind * FLOW_MAX_CHUNKS + c] = un;
    }
  }
}

template <int NV /* dim_h / 128 */>
__global__ void __launch_bounds__(FLOW_THREADS, 1) fmt_flow_kernel(const __grid_constant__ FlowParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ FlowItem items[FLOW_MAX_GEMMS];
  __shared__ FlowChunk chunks[FLOW_MAX_CHUNKS];
  __shared__ FlowUnits units[4 * FLOW_MAX_CHUNKS];
  __shared__ float red_smem[8 * 16];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  FlowSmem sm;
  sm.wring = smem;
  sm.aring = smem + p.nw * FLOW_W_BYTES;
  sm.stg = reinterpret_cast<float*>(sm.aring + p.na * p.a_slot_bytes);
  sm.w_full = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sm.stg) + 2 * FLOW_STG_BYTES);
  sm.w_empty = sm.w_full + FLOW_MAX_NW;
  sm.a_full = sm.w_empty + FLOW_MAX_NW;
  sm.a_empty = sm.a_full + FLOW_MAX_NA;
  sm.t_full = sm.a_empty + FLOW_MAX_NA;
  sm.t_empty = sm.t_full + FLOW_MAX_TS;
  sm.tmem_slot = reinterpret_cast<uint32_t*>(sm.t_empty + FLOW_MAX_TS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nctas = gridDim.x, cta = blockIdx.x;
  // ---- tables: this CTA's item of every GEMM, the chunks, this CTA's units of every (SIMT kind, chunk)
  for (int g = threadIdx.x; g < p.n_gemms; g += FLOW_THREADS) {
    const FlowGemm G = p.gemms[g];
    int item = cta - G.cta_off;
    if (item < 0) item += nctas;
    FlowItem it;
    it.ft = -1; it.kb0 = 0; it.kb1 = 0;
    if (item < G.n_ft * G.pk) {
      const int ft = item % G.n_ft, ks = item / G.n_ft;
      it.kb0 = ks * G.nkb / G.pk; it.kb1 = (ks + 1) * G.nkb / G.pk;
      if (it.kb1 > it.kb0) it.ft = ft;
    }
    it.tm_w = G.tm_w; it.tm_acc = G.tm_acc; it.a_src = G.a_src; it.n_items = G.n_items; it.nkb = G.nkb; it.par_blk = G.par_blk;
    it.pad0 = it.pad1 = it.pad2 = 0;
    items[g] = it;
  }
  flow_chunk_tables<NV>(p, chunks, units, nctas, cta);
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < FLOW_MAX_NW; ++i) { mbar_init(&sm.w_full[i], 1); mbar_init(&sm.w_empty[i], 1); }
    for (int i = 0; i < FLOW_MAX_NA; ++i) { mbar_init(&sm.a_full[i], 1); mbar_init(&sm.a_empty[i], 1); }
    for (int i = 0; i < FLOW_MAX_TS; ++i) { mbar_init(&sm.t_full[i], 1); mbar_init(&sm.t_empty[i], 4); }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(sm.tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *sm.tmem_slot;
  const int n_eval = p.n_steps * p.n_stages;
  if (p.trace != nullptr && threadIdx.x == 96) flow_calibrate(p, 0);     // idle warp 3: SM clock <-> global timer

  // register budget per warpgroup (64 K registers per SM): 64 + 80 + 2 x 184 = 512 per lane quartet
  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
    if (warp == 0) {
      if (lane == 0) flow_weight_producer(p, items, sm, n_eval);
      __syncwarp();
    } else if (warp == 1) {
      if (lane == 0) flow_act_loader(p, items, chunks, units, sm, n_eval);
      __syncwarp();
    } else if (warp == 2) {
      flow_mma_issuer(p, items, sm, tmem_base, n_eval);
    }
  } else if (warp < 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
    flow_epilogue(p, items, chunks, sm, tmem_base, n_eval);
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 184;");
    flow_simt_engine<NV>(p, items, chunks, units, red_smem, n_eval);
  }
  tc_fence_before();
  __syncthreads();
  if (p.trace != nullptr && threadIdx.x == 96) flow_calibrate(p, 1);
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}

}  // namespace fmt
