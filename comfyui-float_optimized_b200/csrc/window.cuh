// Persistent window kernel for the weight-streaming regime (R = nb*B*60 <= 256 token rows, i.e. one or two clips per GPU).
//
// One launch runs EVERY model evaluation of a sampling window (S Euler steps, or S x stages for the RK solvers): 148
// CTAs (one per SM) walk the same list of ~68 stages per evaluation and meet at a grid barrier between stages.
//
//   * GEMM stage   acc[R, N] += A[R, K] . W[N, K]^T   weight-stationary + split-K: item (ft, ks) = 128 output features x a
//                  range of 64-wide K blocks; the weight tile is the UMMA A operand (M = 128), ALL token rows are the UMMA
//                  B operand (N = Rp), so every weight byte is pulled from HBM exactly once by exactly one SM.  The fp32
//                  partial tile goes TMEM -> registers -> smem -> L2 with TMA reduce-add (cp.reduce.async.bulk.tensor), so
//                  split-K costs one pass over the tile and no atomics from the SM.
//   * weight ring  warp 0 is a free-running TMA producer: it walks this CTA's items of ALL stages and evaluations and
//                  keeps an 80 KB ring of weight tiles full.  It never waits for a grid barrier, so the HBM weight stream
//                  keeps flowing while the other warps wait on barriers, activations or epilogues.
//   * SIMT stages  consume the fp32 accumulators and produce the next bf16 operand: ROW (bias, gate, residual, LayerNorm,
//                  AdaLN modulate), ATTN (band attention), GELU, COMB (CFG combine + ODE update).  Each consumer zeroes the
//                  accumulator it has read, so the reduce-add target is clean for the next use.
//
// A stage lasts 4-6 us, so the kernel is written against latency, not throughput (measurements in DESIGN.md section 6):
//   * no local memory - the barrier's ld.acquire.gpu polls are followed by CCTL.IVALL, every spill / stack slot would be
//     re-fetched from L2 after every barrier: one inlined function, 0-byte stack, loop state that does not fit 168 registers
//     lives in shared memory (WinCtx, WinItems, ring positions);
//   * no integer division on the critical path - each CTA's item of every GEMM is tabulated at kernel start;
//   * warp-uniform MMA issue loop with a handful of instructions per K block.
// fmt_window_kernel<NV, true> is a second, experimental schedule of the same stages (one group of CTAs per sequence, N-split
// GEMMs with roles of the UMMA operands swapped, fused GELU): see "GEMM, grouped schedule" below and DESIGN.md section 4a'.
// Reference semantics: FMT.py:151-198 (block / decoder), :277-340 (forward), :342-401 (CFG), torchdiffeq fixed-grid solvers.
#pragma once
#include "kernels.cuh"

namespace fmt {

constexpr int WIN_THREADS = 288;                 // warp 0: weight producer; warps 1..8: main group (256 threads)
constexpr int WIN_MAIN = 256;
constexpr int WIN_NW = 5;                        // weight ring slots
constexpr int WIN_W_BYTES = 128 * 64 * 2;        // one weight tile: 128 features x 64 K, bf16
constexpr int WIN_A_RING = 96 * 1024;            // activation ring: floor(96 KB / (Rp * 128 B)) slots
constexpr int WIN_MAX_NA = 8;
constexpr int WIN_STG_BYTES = 32 * 128 * 4;      // epilogue staging: 32 rows x 128 features fp32
constexpr int WIN_BAR_BYTES = 512;
constexpr int WIN_SMEM_BYTES = WIN_NW * WIN_W_BYTES + WIN_A_RING + 2 * WIN_STG_BYTES + WIN_BAR_BYTES + 1024;
// grouped schedule: every CTA pulls 1/Cg (not 1/148) of a layer's weights plus the whole operand of its group per stage, and the
// rate of that pull is (bytes in flight) / (L2 or HBM latency): the rings take all of shared memory and a weight slot holds
// several K blocks (24 KB / (nf * 128 B)), so ~144 KB of weights are requested before the stage starts
// Slots hold SEVERAL K blocks (weights: 24 KB / (nf * 128 B); activations: 32 KB / (RgP * 128 B)): a slot is handed back with
// ONE tcgen05.commit, and commits are the expensive part of the hand-off (measured: a loop that commits twice per K block
// paces at ~0.45 us per K block with no loads and no MMAs in flight).
constexpr int WIN2_NW = 4;
constexpr int WIN2_W_BYTES = 24 * 1024;
constexpr int WIN2_NA = 3;
constexpr int WIN2_A_BYTES = 32 * 1024;          // 4 K blocks of a 64-row group, 2 of a 128-row group
constexpr int WIN2_A_RING = WIN2_NA * WIN2_A_BYTES + 8 * 1024;   // + 8 KB the M = 128 descriptor of the last K block reaches into when RgP = 64
constexpr int WIN2_SMEM_BYTES = WIN2_NW * WIN2_W_BYTES + WIN2_A_RING + WIN_BAR_BYTES + 1024;
constexpr int WIN_MAX_DEPTH = 16;
constexpr int WIN_MAX_GEMMS = 2 + 4 * WIN_MAX_DEPTH;

struct WinGemm {
  int tm_w, tm_a, tm_acc;   // tensor-map indices: weights (box 64 x 128), activations (box 64 x Rp), accumulator (box 128 x 32, fp32)
  int n_ft;                 // ceil(N / 128) feature tiles
  int nkb;                  // ceil(K / 64) K blocks
  int pk;                   // K splits; n_ft * pk <= gridDim.x items, item i runs on CTA (i + cta_off) % gridDim.x
  int cta_off;
  int a_tiled;              // 1: the activation operand is stored pre-tiled (see win_tiled_off) and fetched with plain bulk copies; tm_a = buffer id
  // grouped schedule (fmt_window_kernel<NV, true>): item = nf output features x a range of K blocks, one item per CTA of a group
  int nf;                   // output features per item (multiple of 16, <= 128) = UMMA N
  int n_nt;                 // ceil(N / nf) feature slices
  int N;                    // output features of the layer
  int out;                  // 0: Pacc, 1: QKVacc, 2: Hacc, 3: Vacc
  int epi;                  // 0: accumulator (+)= partial; 1: Hm = bf16(GELU(acc + bias)) (fc1 with pk == 1: the GELU stage is skipped)
};

// Operand layout of A1 / A2 / Hm inside the window kernel: [K block][Rp rows][64 bf16] with the 128-byte swizzle of the UMMA
// descriptor already applied (16-byte chunk index XOR row mod 8), i.e. each K block is the exact shared-memory image of a
// SW128 K-major tile and is fetched with ONE contiguous cp.async.bulk (measured 165-205 GB/s per SM against ~70 GB/s for
// the 2D tensor-map load whose rows are 128-byte fragments 2 KB apart).  Rows >= R are never written and stay zero.
__device__ __forceinline__ size_t win_tiled_off(int r, int c, int Rp) {       // element offset of (row r, column c); c % 4 == 0 keeps 4 elements contiguous
  const int kb = c >> 6, cc = c & 63;
  return static_cast<size_t>(kb) * Rp * 64 + static_cast<size_t>(r) * 64 + ((((cc >> 3) ^ (r & 7)) << 3) | (cc & 7));
}

struct WinParams {
  ModelShape s;
  int R, Rp, depth, heads, window, mlp_hidden, NT;
  int n_steps, n_stages, n_gemms;
  WinGemm gemms[WIN_MAX_GEMMS];        // x_emb, (qkv, proj, fc1, fc2) x depth, dec
  const CUtensorMap* tmaps;            // device array
  float *X, *Pacc, *QKVacc, *Hacc, *Vacc;
  __nv_bfloat16 *A1, *A2, *Hm, *ax;
  const __nv_bfloat16* table;          // (n_eval, R, NT)
  const float *b_x, *pos, *b_dec;
  const float *b_qkv[WIN_MAX_DEPTH], *b_proj[WIN_MAX_DEPTH], *b_fc1[WIN_MAX_DEPTH], *b_fc2[WIN_MAX_DEPTH];
  float *x_state, *kbuf;
  const float* ddt;
  float rk_a[16], rk_b[4];
  const WindowArgs* wargs;
  unsigned* bar_counter;               // zeroed before every launch
  int* err_flag;
  long long* trace;                    // optional (FMT_WIN_TRACE=1): [cta][barrier][6] SM-clock stamps (arrive, pass, 4 intra-stage marks of the NEXT stage)
  int trace_stride;                    // barriers per CTA recorded
  int w_lookahead;                     // weight prefetch may run this many stages ahead of the stage in flight (>= 1000: ungated)
  // grouped schedule: G groups of Cg CTAs, group g owns token rows [g * Rg, (g + 1) * Rg) (whole sequences) and its own
  // pre-tiled operand buffers of RgP (64 or 128) rows; bar_counter[32 * (1 + g)] is the group's barrier, bar_counter[0] the global one
  int G, Cg, Rg, RgP;
  int fuse_gelu;                       // 1: fc1's epilogue writes Hm, evaluation has 4 + 7 * depth stages
};

// What a CTA works on in the SIMT stages: all rows / all CTAs in the split-K schedule, one group's rows / CTAs in the grouped one.
struct WinCtx {
  int row0, nrows;                     // token rows [row0, row0 + nrows)
  int rank, nranks;                    // this CTA among the CTAs sharing those rows
  int all_rank, all_n;                 // this CTA among all working CTAs (COMB stage)
  int RgP;                             // padded rows of the pre-tiled operand buffers below
  __nv_bfloat16 *A1, *A2, *Hm;         // this group's pre-tiled operands (local row = r - row0)
  unsigned* bar;                       // the barrier counter shared by `nranks` CTAs
};

// ---------------------------------------------------------------- small PTX helpers local to this kernel
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async.global;" ::: "memory"); }   // measured: 100 cycles vs 590 for the all-space form
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* m, const void* smem_src, int32_t crd0, int32_t crd1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(crd0), "r"(crd1)
               : "memory");
}
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)), "l"(src), "r"(bytes),
               "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_gpu_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Bounded spins: a protocol bug must end in a trap (reported as a launch failure), never in a hung GPU.
constexpr long long WIN_SPIN_LIMIT = 4000000000ll;   // ~2 s of SM clocks
__device__ __forceinline__ void win_fail(int* err_flag, int code) {
  if (err_flag != nullptr) atomicExch(err_flag, code);
  __threadfence_system();
  __trap();
}
__device__ __forceinline__ void mbar_wait_b(uint64_t* bar, uint32_t parity, int* err_flag, int code) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > WIN_SPIN_LIMIT) win_fail(err_flag, code);
  }
}

// intra-stage mark `slot` (0..3) of the stage that follows barrier `epoch` (call from ONE thread per CTA and slot)
__device__ __forceinline__ void win_mark(const WinParams& p, unsigned epoch, int slot) {
  if (p.trace != nullptr && epoch >= 1 && static_cast<int>(epoch) <= p.trace_stride)
    p.trace[(static_cast<size_t>(blockIdx.x) * p.trace_stride + (epoch - 1)) * 6 + 2 + slot] = clock64();
}

struct WinSmem {
  uint8_t* wring;
  uint8_t* aring;
  float* stg;
  uint64_t *w_full, *w_empty, *a_full, *a_empty, *t_full;
  uint32_t* tmem_slot;
  int* gate;          // quiet points passed (see win_weight_producer)
  int nw, w_bytes;    // weight ring: slots, bytes per slot
};

// barrier over the CTAs that share `counter` (the whole grid, or one group), entered by the main group (256 threads, named
// barrier 1).  ctr[] lives in shared memory (a register copy would be spilled, and a spill costs an L2 round trip per barrier):
// ctr[0] = barriers this CTA has passed (trace index), ctr[which] = barriers passed on this counter; `nranks` arrivals complete one;
// ctr[3] = evaluations finished.
__device__ __forceinline__ void win_grid_sync(const WinParams& p, volatile unsigned* ctr, unsigned* counter, int which, unsigned nranks,
                                              bool end_of_eval) {
  fence_proxy_async_all();                 // this thread's generic-proxy writes -> visible to later TMA (async proxy) reads
  named_bar_sync(1, WIN_MAIN);
  if (threadIdx.x == 32) {
    const unsigned epoch = ctr[0] + 1, target = (ctr[which] + 1) * nranks;
    ctr[0] = epoch; ctr[which] = ctr[which] + 1;
    if (end_of_eval) ctr[3] = ctr[3] + 1;  // evaluations finished (the loop counter of the kernel, kept out of the register file too)
    long long* tr = (p.trace != nullptr && static_cast<int>(epoch) <= p.trace_stride)
                        ? p.trace + (static_cast<size_t>(blockIdx.x) * p.trace_stride + (epoch - 1)) * 6 : nullptr;
    if (tr) tr[0] = clock64();
    red_release_gpu_add(counter, 1u);
    const long long t0 = clock64();
    // acquire loads, back to back.  Measured alternative: relaxed polls (with 0-200 ns pauses) and one fence.acq_rel.gpu after the
    // last one avoid the CCTL.IVALL per poll but cost 25 us per ODE step more - the full fence drains this SM's outstanding writes.
    while (ld_acquire_gpu(counter) < target) {
      if (clock64() - t0 > WIN_SPIN_LIMIT) win_fail(p.err_flag, 100 + static_cast<int>(epoch & 0xffff));
    }
    if (tr) tr[1] = clock64();
  }
  named_bar_sync(1, WIN_MAIN);
}

__device__ __forceinline__ bool win_item(const WinGemm& G, int& ft, int& kb0, int& kb1) {
  int item = static_cast<int>(blockIdx.x) - G.cta_off;
  if (item < 0) item += gridDim.x;
  if (item >= G.n_ft * G.pk) return false;
  ft = item % G.n_ft;
  const int ks = item / G.n_ft;
  kb0 = ks * G.nkb / G.pk;
  kb1 = (ks + 1) * G.nkb / G.pk;
  return kb1 > kb0;
}

struct WinRing {   // ring position kept identically by every lane of a role warp
  int w_slot = 0; uint32_t w_phase = 0;
  int a_slot = 0; uint32_t a_phase = 0;
  uint32_t t_phase = 0;
};

// This CTA's item of every GEMM, computed once at kernel start (the integer divisions of win_item / win_item2 cost ~0.5 us per
// stage when a single warp executes them on the critical path): x = feature tile / slice (-1: no item), y = first K block, z = end
struct WinItems { int4 it[WIN_MAX_GEMMS]; };

// ---------------------------------------------------------------------------------------------------------------- GEMM
__device__ __forceinline__ void win_gemm_stage(const WinParams& p, const WinGemm& G, const int4 item, const WinSmem& sm, WinRing& rg, int NA,
                                               uint32_t tmem_base, unsigned epoch) {
  if (item.x < 0) {
    if (threadIdx.x == 32) atomicAdd_block(sm.gate, 1);
    return;
  }
  const int ft = item.x, kb0 = item.y, kb1 = item.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, mw = warp - 1;
  const int a_bytes = p.Rp * 128;
  if (mw == 0) {
    // ===================== activation producer =====================
    for (int kb = kb0; kb < kb1; ++kb) {
      if (lane == 0) {
        mbar_wait_b(&sm.a_empty[rg.a_slot], rg.a_phase ^ 1, p.err_flag, 1);
        mbar_expect_tx(&sm.a_full[rg.a_slot], a_bytes);
        if (G.a_tiled) {
          const __nv_bfloat16* src = (G.tm_a == 0 ? p.A1 : G.tm_a == 1 ? p.A2 : p.Hm) + static_cast<size_t>(kb) * p.Rp * 64;
          bulk_load_1d(sm.aring + rg.a_slot * a_bytes, src, a_bytes, &sm.a_full[rg.a_slot]);
        } else {
          tma_load_2d(&p.tmaps[G.tm_a], &sm.a_full[rg.a_slot], sm.aring + rg.a_slot * a_bytes, kb * 64, 0, kEvictLast);
        }
      }
      if (++rg.a_slot == NA) { rg.a_slot = 0; rg.a_phase ^= 1; }
    }
    __syncwarp();
  } else if (mw == 1) {
    // ===================== MMA issuer =====================
    // warp-uniform loop (every lane waits, one elected lane issues) with a small body: a single warp runs dependent
    // instructions at ~5 cycles each, so at 4 MMAs per K block the instruction count of this loop paces the stage
    const uint32_t idesc = make_idesc_bf16_f32(128, static_cast<uint32_t>(p.Rp));
    const uint64_t desc_hi = make_sw128_kmajor_desc(0);
    const uint32_t w_base = smem_u32(sm.wring) >> 4, a_base = smem_u32(sm.aring) >> 4, ab16 = a_bytes >> 4;
    const bool leader = elect_one();
    int w_slot = rg.w_slot, a_slot = rg.a_slot;
    uint32_t w_phase = rg.w_phase, a_phase = rg.a_phase;
    uint32_t accum = 0;
    for (int kb = kb0; kb < kb1; ++kb) {
      mbar_wait_b(&sm.w_full[w_slot], w_phase, p.err_flag, 2);
      mbar_wait_b(&sm.a_full[a_slot], a_phase, p.err_flag, 3);
      tc_fence_after();
      if (leader) {
        const bool last = kb == kb1 - 1;
        const uint64_t dw = desc_hi | (w_base + w_slot * (WIN_W_BYTES >> 4)), da = desc_hi | (a_base + a_slot * ab16);
        umma_bf16(tmem_base, dw, da, idesc, accum);
        umma_bf16(tmem_base, dw + 2, da + 2, idesc, 1u);
        umma_bf16(tmem_base, dw + 4, da + 4, idesc, 1u);
        umma_bf16(tmem_base, dw + 6, da + 6, idesc, 1u);
        umma_commit(&sm.w_empty[w_slot]);
        umma_commit(&sm.a_empty[a_slot]);
        if (last) { umma_commit(sm.t_full); atomicAdd_block(sm.gate, 1); win_mark(p, epoch, 0); }   // quiet point: this stage's operands have landed
      }
      accum = 1u;
      if (++w_slot == WIN_NW) { w_slot = 0; w_phase ^= 1; }
      if (++a_slot == NA) { a_slot = 0; a_phase ^= 1; }
    }
    rg.w_slot = w_slot; rg.w_phase = w_phase; rg.a_slot = a_slot; rg.a_phase = a_phase;
    __syncwarp();
  } else if (mw >= 4) {
    // ===================== epilogue: TMEM (lanes = features, columns = rows) -> smem [row][feature] -> L2 reduce-add
    const int quarter = warp & 3;
    const int fl = quarter * 32 + lane;
    const bool issuer = (mw == 4 && lane == 0);
    if (lane == 0) mbar_wait_b(sm.t_full, rg.t_phase, p.err_flag, 4);      // one poller per warp
    __syncwarp();
    rg.t_phase ^= 1;
    tc_fence_after();
    if (issuer) win_mark(p, epoch, 1);
    // One SM's TMA write path drains a 16 KB chunk in ~0.37 us (2.25 us for the 98 KB tile) whatever the other SMs do - the same
    // with 148, 64 or 32 CTAs reducing, the same with plain TMA stores instead of reduce-adds, and a second team of four warps
    // feeding the engine from its own staging buffer made it slower (2.9 us).  The LSU is slower still: scalar red.global.add.f32
    // straight from the TMEM registers (one 128-byte line per warp instruction) 5.1 us, red.global.add.v4.f32 from the staging
    // buffer (one 512-byte tile row per warp instruction) 4.6 us; handing the last one / two / three chunks to the idle warps
    // 1-4 as LSU reds while warps 5-8 feed the TMA path: 355 / 361 / 399 us per ODE step against 356.
    const int n_chunks = (p.R + 31) / 32;
    for (int c = 0; c < n_chunks; ++c) {
      float* stg = sm.stg + (c & 1) * (WIN_STG_BYTES / 4);
      float v[32];
      tmem_ld32(tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + c * 32, v);
      if (c >= 2) {                       // the reduce that read this staging buffer two chunks ago must be done reading
        if (issuer) bulk_wait_read<1>();
        named_bar_sync(2, 128);
      }
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) stg[j * 128 + fl] = v[j];
      fence_proxy_async();                // smem writes -> visible to the async proxy
      named_bar_sync(2, 128);
      if (issuer) {
        tma_reduce_add_2d(&p.tmaps[G.tm_acc], stg, ft * 128, c * 32);
        bulk_commit();
      }
    }
    if (issuer) {
      win_mark(p, epoch, 2);
      bulk_wait<0>();                     // all partial sums are in L2 before this CTA arrives at the grid barrier
      win_mark(p, epoch, 3);
    }
    tc_fence_before();
  }
}

// ------------------------------------------------------------------------------------------------- GEMM, grouped schedule
// Group g (Cg CTAs) owns whole sequences: <= 128 token rows.  Roles are swapped with respect to the split-K schedule: the
// group's activation tile [RgP rows x 64 K] is the UMMA A operand (M = 128; with RgP = 64 the upper 64 lanes read whatever
// follows in the ring and are never looked at), the weight slice [nf features x 64 K] is the B operand (N = nf), so the
// output features of a layer are dealt to the CTAs of the group in slices of nf (a multiple of 16, not of 128) and K is
// split at most pk <= 4 ways.  The fp32 tile D[row = TMEM lane, feature = column] leaves through registers: pk == 1 ->
// plain 256-bit stores (or the fused GELU -> bf16 operand), pk > 1 -> red.global.add.v4.f32 (64 rows x nf x 4 B per CTA).
__device__ __forceinline__ bool win_item2(const WinGemm& G, const WinCtx& cx, int& nt, int& kb0, int& kb1) {
  int item = cx.rank - G.cta_off;
  if (item < 0) item += cx.nranks;
  if (item >= G.n_nt * G.pk) return false;
  nt = item % G.n_nt;
  const int ks = item / G.n_nt;
  kb0 = ks * G.nkb / G.pk;
  kb1 = (ks + 1) * G.nkb / G.pk;
  return kb1 > kb0;
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ float gelu_tanh_fast(float x);

__device__ __forceinline__ void win_gemm2_stage(const WinParams& p, const WinCtx& cx, const WinGemm& G, const int4 item, const WinSmem& sm, WinRing& rg,
                                                uint32_t tmem_base, unsigned epoch, const float* __restrict__ bias) {
  if (item.x < 0) {
    if (threadIdx.x == 32) atomicAdd_block(sm.gate, 1);
    return;
  }
  const int nt = item.x, kb0 = item.y, kb1 = item.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, mw = warp - 1;
  const int a_bytes = cx.RgP * 128;
  if (mw == 0) {
    // ===================== activation producer: this group's K blocks kb0..kb1 of the operand, kpa per ring slot =====================
    const int kpa = WIN2_A_BYTES / a_bytes;
    for (int kb = kb0; kb < kb1; kb += kpa) {
      const int n = min(kpa, kb1 - kb);
      if (lane == 0) {
        uint8_t* dst = sm.aring + rg.a_slot * WIN2_A_BYTES;
        mbar_wait_b(&sm.a_empty[rg.a_slot], rg.a_phase ^ 1, p.err_flag, 1);
        mbar_expect_tx(&sm.a_full[rg.a_slot], n * a_bytes);
        if (G.a_tiled) {      // consecutive K blocks of the pre-tiled operand are contiguous: one bulk copy per slot
          const __nv_bfloat16* src = (G.tm_a == 0 ? cx.A1 : G.tm_a == 1 ? cx.A2 : cx.Hm) + static_cast<size_t>(kb) * cx.RgP * 64;
          bulk_load_1d(dst, src, n * a_bytes, &sm.a_full[rg.a_slot]);
        } else {   // row-major x-embedder operand: box = 64 K x RgP rows starting at the group's first row (rows past R are zero-filled)
          for (int j = 0; j < n; ++j) tma_load_2d(&p.tmaps[G.tm_a], &sm.a_full[rg.a_slot], dst + j * a_bytes, (kb + j) * 64, cx.row0, kEvictLast);
        }
      }
      if (++rg.a_slot == WIN2_NA) { rg.a_slot = 0; rg.a_phase ^= 1; }
    }
    __syncwarp();
  } else if (mw == 1) {
    // ===================== MMA issuer: D[128 x nf] += A[128 x 16] . W[nf x 16]^T =====================
    // The loop is warp-uniform (every lane waits, one elected lane issues) and keeps its per-K-block instruction count low: a
    // single warp runs it at ~5 cycles per dependent instruction, and at 4 small MMAs per K block that, not the tensor pipe,
    // sets the pace (measured 0.45 us per K block with ~150 instructions in the body).
    const uint32_t idesc = make_idesc_bf16_f32(128, static_cast<uint32_t>(G.nf));
    const int tile = G.nf * 128, kps = WIN2_W_BYTES / tile;              // K blocks per weight slot (same chunking as the producer)
    const int kpa = WIN2_A_BYTES / a_bytes;                              // K blocks per activation slot
    const uint64_t desc_hi = make_sw128_kmajor_desc(0);
    const uint32_t w_base = smem_u32(sm.wring) >> 4, a_base = smem_u32(sm.aring) >> 4;
    const uint32_t tile16 = tile >> 4, ab16 = a_bytes >> 4;
    const bool leader = elect_one();
    int w_slot = rg.w_slot, a_slot = rg.a_slot;
    uint32_t w_phase = rg.w_phase, a_phase = rg.a_phase;
    int j = 0, ja = 0;
    uint32_t wa = w_base + w_slot * (WIN2_W_BYTES >> 4), aa = a_base + a_slot * (WIN2_A_BYTES >> 4);
    uint32_t accum = 0;
    for (int kb = kb0; kb < kb1; ++kb) {
      const bool last = kb == kb1 - 1;
      if (j == 0) mbar_wait_b(&sm.w_full[w_slot], w_phase, p.err_flag, 2);
      if (ja == 0) mbar_wait_b(&sm.a_full[a_slot], a_phase, p.err_flag, 3);
      tc_fence_after();
      const bool w_done = (++j == kps) || last, a_done = (++ja == kpa) || last;
      if (leader) {
        if (kb == kb0) win_mark(p, epoch, 0);                            // first operands landed
        const uint64_t dw = desc_hi | wa, da = desc_hi | aa;
        umma_bf16(tmem_base, da, dw, idesc, accum);
        umma_bf16(tmem_base, da + 2, dw + 2, idesc, 1u);
        umma_bf16(tmem_base, da + 4, dw + 4, idesc, 1u);
        umma_bf16(tmem_base, da + 6, dw + 6, idesc, 1u);
        if (w_done) umma_commit(&sm.w_empty[w_slot]);
        if (a_done) umma_commit(&sm.a_empty[a_slot]);
        if (last) { umma_commit(sm.t_full); atomicAdd_block(sm.gate, 1); win_mark(p, epoch, 1); }   // quiet point: this stage's operands have landed
      }
      accum = 1u;
      wa += tile16; aa += ab16;
      if (w_done) { j = 0; if (++w_slot == WIN2_NW) { w_slot = 0; w_phase ^= 1; } wa = w_base + w_slot * (WIN2_W_BYTES >> 4); }
      if (a_done) { ja = 0; if (++a_slot == WIN2_NA) { a_slot = 0; a_phase ^= 1; } aa = a_base + a_slot * (WIN2_A_BYTES >> 4); }
    }
    rg.w_slot = w_slot; rg.w_phase = w_phase; rg.a_slot = a_slot; rg.a_phase = a_phase;
    __syncwarp();
  } else if (mw >= 4) {
    // ===================== epilogue: lane = token row, columns = this item's features =====================
    const int quarter = warp & 3;
    if (lane == 0) mbar_wait_b(sm.t_full, rg.t_phase, p.err_flag, 4);      // one poller per warp
    __syncwarp();
    rg.t_phase ^= 1;
    tc_fence_after();
    if (quarter == 0 && lane == 0) win_mark(p, epoch, 2);
    if (quarter * 32 < cx.RgP) {
      const int lr = quarter * 32 + lane;
      const bool valid = lr < cx.nrows;
      const int f0 = nt * G.nf;
      float* acc = (G.out == 0 ? p.Pacc : G.out == 1 ? p.QKVacc : G.out == 2 ? p.Hacc : p.Vacc) + static_cast<size_t>(cx.row0 + lr) * G.N + f0;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
      const int ncol = min(G.nf, G.N - f0);                              // valid columns (multiple of 16)
#pragma unroll 1
      for (int c = 0; c < ncol; c += 16) {
        float v[16];
        tmem_ld16(taddr + c, v);
        tmem_ld_wait();
        if (!valid) continue;
        if (G.epi == 1) {
          // fc1: Hm = bf16(GELU(acc + b)), written as 16-byte chunks of the pre-tiled operand (FMT.py:159-162)
#pragma unroll
          for (int j = 0; j < 16; j += 8) {
            const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + f0 + c + j)), b1 = __ldg(reinterpret_cast<const float4*>(bias + f0 + c + j + 4));
            uint4 t;
            t.x = pack_bf16x2(gelu_tanh_fast(v[j] + b0.x), gelu_tanh_fast(v[j + 1] + b0.y));
            t.y = pack_bf16x2(gelu_tanh_fast(v[j + 2] + b0.z), gelu_tanh_fast(v[j + 3] + b0.w));
            t.z = pack_bf16x2(gelu_tanh_fast(v[j + 4] + b1.x), gelu_tanh_fast(v[j + 5] + b1.y));
            t.w = pack_bf16x2(gelu_tanh_fast(v[j + 6] + b1.z), gelu_tanh_fast(v[j + 7] + b1.w));
            *reinterpret_cast<uint4*>(cx.Hm + win_tiled_off(lr, f0 + c + j, cx.RgP)) = t;
          }
        } else if (G.pk == 1) {
#pragma unroll
          for (int j = 0; j < 16; j += 8)
            st_global_v8(acc + c + j, __float_as_uint(v[j]), __float_as_uint(v[j + 1]), __float_as_uint(v[j + 2]), __float_as_uint(v[j + 3]),
                         __float_as_uint(v[j + 4]), __float_as_uint(v[j + 5]), __float_as_uint(v[j + 6]), __float_as_uint(v[j + 7]));
        } else {
#pragma unroll
          for (int j = 0; j < 16; j += 4) red_add_v4(acc + c + j, v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      }
      if (quarter == 0 && lane == 0) win_mark(p, epoch, 3);
    }
    tc_fence_before();
  }
}

// weight producer of the grouped schedule (warp 0): the same free-running ring, items from win_item2
__device__ __forceinline__ void win_weight_producer2(const WinParams& p, const WinItems& items, const WinSmem& sm, int n_eval) {
  int slot = 0; uint32_t phase = 0;
  const int bs = p.fuse_gelu ? 7 : 8;
  const int spe = 4 + bs * p.depth;                    // stages per evaluation
  for (int e = 0; e < n_eval; ++e) {
    for (int g = 0; g < p.n_gemms; ++g) {
      const WinGemm& G = p.gemms[g];
      const int4 item = items.it[g];
      if (item.x < 0) continue;
      const int nt = item.x, kb0 = item.y, kb1 = item.z;
      // stage index of GEMM g inside an evaluation: 0 | 2 + bs * blk + {0 qkv, 2 proj, 4 fc1, 6 (5 when GELU is fused) fc2} | spe - 2
      const int q = (g - 1) % 4;
      const int si = g == 0 ? 0 : (g == p.n_gemms - 1 ? spe - 2 : 2 + bs * ((g - 1) / 4) + (q == 3 && p.fuse_gelu ? 5 : 2 * q));
      const int need = e * spe + si - p.w_lookahead + 1;
      if (need > 0) {
        const long long t0 = clock64();
        while (*reinterpret_cast<volatile int*>(sm.gate) < need) {
          __nanosleep(64);
          if (clock64() - t0 > WIN_SPIN_LIMIT) win_fail(p.err_flag, 6);
        }
      }
      const int tile = G.nf * 128, kps = WIN2_W_BYTES / tile;            // K blocks per ring slot
      for (int kb = kb0; kb < kb1; kb += kps) {
        const int n = min(kps, kb1 - kb);
        mbar_wait_b(&sm.w_empty[slot], phase ^ 1, p.err_flag, 5);
        mbar_expect_tx(&sm.w_full[slot], n * tile);
        for (int j = 0; j < n; ++j)
          tma_load_2d(&p.tmaps[G.tm_w], &sm.w_full[slot], sm.wring + slot * WIN2_W_BYTES + j * tile, (kb + j) * 64, nt * G.nf, kEvictNormal);
        if (++slot == WIN2_NW) { slot = 0; phase ^= 1; }
      }
    }
  }
}

// W-producer's view of the same item list (warp 0, free-running over the whole window)
// Gating: the refill of the ring competes with the latency-critical loads of the stage in flight (measured: a SIMT stage's
// L2 loads take 1.5 us instead of 0.65 us while 148 producers burst), so the weights of global stage s may only be
// requested once `gate` (quiet points passed = stages whose own loads have landed) has reached s - w_lookahead + 1.
__device__ __forceinline__ void win_weight_producer(const WinParams& p, const WinItems& items, const WinSmem& sm, int n_eval) {
  int slot = 0; uint32_t phase = 0;
  const int spe = 4 + 8 * p.depth;                     // stages per evaluation
  for (int e = 0; e < n_eval; ++e) {
    for (int g = 0; g < p.n_gemms; ++g) {
      const WinGemm& G = p.gemms[g];
      const int4 item = items.it[g];
      if (item.x < 0) continue;
      const int ft = item.x, kb0 = item.y, kb1 = item.z;
      const int si = g == 0 ? 0 : (g == p.n_gemms - 1 ? spe - 2 : 2 + 8 * ((g - 1) / 4) + 2 * ((g - 1) % 4));
      const int need = e * spe + si - p.w_lookahead + 1;
      if (need > 0) {
        const long long t0 = clock64();
        while (*reinterpret_cast<volatile int*>(sm.gate) < need) {
          __nanosleep(64);
          if (clock64() - t0 > WIN_SPIN_LIMIT) win_fail(p.err_flag, 6);
        }
      }
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait_b(&sm.w_empty[slot], phase ^ 1, p.err_flag, 5);
        mbar_expect_tx(&sm.w_full[slot], WIN_W_BYTES);
        tma_load_2d(&p.tmaps[G.tm_w], &sm.w_full[slot], sm.wring + slot * WIN_W_BYTES, kb * 64, ft * 128, kEvictFirst);
        if (++slot == WIN_NW) { slot = 0; phase ^= 1; }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------- SIMT
// Every SIMT stage is latency-bound (one L2 round trip is ~0.8 us, a stage has microseconds): all global loads of a work
// item are issued before the first dependent instruction, and nothing is stored before the last load has been issued.
__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void bf16x4_to_f32(uint2 t, float (&v)[4]) {
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&t.x), b = *reinterpret_cast<__nv_bfloat162*>(&t.y);
  v[0] = __low2float(a); v[1] = __high2float(a); v[2] = __low2float(b); v[3] = __high2float(b);
}
__device__ __forceinline__ uint2 f32x4_to_bf16(const float (&v)[4]) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
  uint2 t;
  t.x = *reinterpret_cast<uint32_t*>(&a);
  t.y = *reinterpret_cast<uint32_t*>(&b);
  return t;
}
__device__ __forceinline__ uint2 ld_nc_u2(const __nv_bfloat16* p) { return __ldg(reinterpret_cast<const uint2*>(p)); }

// ROW stage.  WPR warps share one token row (FPL float4 per lane each); rows are dealt round-robin to CTAs.
//   mode 0 (after x_embedder): X = acc + bias + pos_embed[frame]                       (FMT.py:319-320)
//   mode 1 (after proj / fc2): X = X + gate * (acc + bias)                             (FMT.py:174-175)
// then A1 = bf16( LayerNorm(X) * (1 + scale) + shift )  with this evaluation's table row  (FMT.py:168-169,174-175,197)
// and the accumulator row (plus, after proj, the QKV accumulator row) is zeroed for its next use.
template <int NV>
__device__ __forceinline__ void win_row_stage(const WinParams& p, const WinCtx& cx, float* red_smem, const __nv_bfloat16* __restrict__ table_e, int mode,
                                              const float* __restrict__ bias, long long gate_off, long long shift_off, long long scale_off,
                                              bool zero_qkv) {
  constexpr int WPR = NV >= 4 ? 4 : NV;          // warps per row
  constexpr int FPL = NV / WPR;                  // float4 per lane
  constexpr int GROUPS = 8 / WPR;                // rows in flight per CTA
  const int lane = threadIdx.x & 31, mw = (threadIdx.x >> 5) - 1;
  const int grp = mw / WPR, wq = mw % WPR;
  const int H = p.s.H;
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int r = cx.row0 + cx.rank + cx.nranks * grp; r < cx.row0 + cx.nrows; r += cx.nranks * GROUPS) {
    const int c0 = wq * (FPL * 128) + lane * 4;                       // first column of this lane; + i*128 per float4
    float* acc = p.Pacc + static_cast<size_t>(r) * H + c0;
    float* xr = p.X + static_cast<size_t>(r) * H + c0;
    const __nv_bfloat16* trow = table_e + static_cast<size_t>(r) * p.NT + c0;
    float4 a[FPL], x[FPL], b[FPL], ps[FPL];
    uint2 tg[FPL], tsh[FPL], tsc[FPL];
#pragma unroll
    for (int i = 0; i < FPL; ++i) {
      a[i] = ldcg4(acc + i * 128);
      tsh[i] = ld_nc_u2(trow + shift_off + i * 128);
      tsc[i] = ld_nc_u2(trow + scale_off + i * 128);
      b[i] = __ldg(reinterpret_cast<const float4*>(bias + c0 + i * 128));
      if (mode == 1) {
        x[i] = ldcg4(xr + i * 128);
        tg[i] = ld_nc_u2(trow + gate_off + i * 128);
      } else {
        ps[i] = __ldg(reinterpret_cast<const float4*>(p.pos + static_cast<size_t>(r % p.s.N) * H + c0 + i * 128));
      }
    }
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
    if (zero_qkv) {
      float* q = p.QKVacc + static_cast<size_t>(r) * 3 * H + wq * (3 * FPL * 128) + lane * 4;
#pragma unroll
      for (int i = 0; i < 3 * FPL; ++i) *reinterpret_cast<float4*>(q + i * 128) = zero4;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (WPR > 1) {
      if (lane == 0) red_smem[mw] = sum;
      named_bar_sync(3 + grp, WPR * 32);
      sum = 0.f;
#pragma unroll
      for (int w = 0; w < WPR; ++w) sum += red_smem[grp * WPR + w];
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
      if (lane == 0) red_smem[8 + mw] = var;
      named_bar_sync(3 + grp, WPR * 32);
      var = 0.f;
#pragma unroll
      for (int w = 0; w < WPR; ++w) var += red_smem[8 + grp * WPR + w];
    }
    const float rstd = rsqrtf(var / static_cast<float>(H) + 1e-6f);
#pragma unroll
    for (int i = 0; i < FPL; ++i) {
      float sh[4], sc[4];
      bf16x4_to_f32(tsh[i], sh);
      bf16x4_to_f32(tsc[i], sc);
      float v[4] = {(x[i].x - mean) * rstd, (x[i].y - mean) * rstd, (x[i].z - mean) * rstd, (x[i].w - mean) * rstd};
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] = fmaf(v[k], 1.f + sc[k], sh[k]);
      *reinterpret_cast<uint2*>(cx.A1 + win_tiled_off(r - cx.row0, c0 + i * 128, cx.RgP)) = f32x4_to_bf16(v);
    }
    if (WPR > 1) named_bar_sync(3 + grp, WPR * 32);   // red_smem is reused by the next row of this group
  }
}

// ATTN stage: band-masked attention (FMT.py:15-19,69-88) straight from the fp32 QKV accumulator (+ qkv bias); one warp
// per (sequence, head, query row), TWO units interleaved per warp so their loads are in flight together.
// Output A2 bf16 = operand of the proj GEMM.
template <int VPL> struct F32Vec;
template <> struct F32Vec<1> { static __device__ __forceinline__ void ld(const float* p, float (&v)[1]) { v[0] = __ldcg(p); } };
template <> struct F32Vec<2> { static __device__ __forceinline__ void ld(const float* p, float (&v)[2]) { float2 t = __ldcg(reinterpret_cast<const float2*>(p)); v[0] = t.x; v[1] = t.y; } };
template <> struct F32Vec<4> { static __device__ __forceinline__ void ld(const float* p, float (&v)[4]) { float4 t = __ldcg(reinterpret_cast<const float4*>(p)); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; } };

// Fast path (band of at most 5 keys = attention_window <= 2): U units per warp, all loads first, plain (not online) softmax.
template <int VPL, int U /* units interleaved per warp */>
__device__ __forceinline__ void win_attn_band5(const WinParams& p, const WinCtx& cx, const float* __restrict__ bqkv) {
  const int lane = threadIdx.x & 31, mw = (threadIdx.x >> 5) - 1;
  constexpr int hd = VPL * 32, KB = 5;
  const int N = p.s.N, heads = p.heads, H = p.s.H, ld = 3 * H;
  const int n_units = cx.nrows * heads;
  const float scale = rsqrtf(static_cast<float>(hd));
  const int win = p.window;
  const int stride = cx.nranks * 8;
  // index arithmetic without runtime divisions on the critical path (a single warp pays ~150 cycles for each)
  const bool h_pow2 = (heads & (heads - 1)) == 0;
  const int h_shift = __ffs(heads) - 1;
  const int sq0 = cx.row0 / N, fi0 = cx.row0 - sq0 * N;      // once per stage
#pragma unroll 1
  for (int u0 = cx.rank + cx.nranks * mw; u0 < n_units; u0 += U * stride) {
    int row[U], hh[U], j0[U], nk[U];
    bool valid[U];
    float q[U][VPL], kv[U][KB][VPL], vv[U][KB][VPL];
#pragma unroll
    for (int t = 0; t < U; ++t) {
      const int u = u0 + t * stride;
      valid[t] = u < n_units;
      const int uu = valid[t] ? u : u0;
      const int lr = h_pow2 ? (uu >> h_shift) : uu / heads;
      hh[t] = h_pow2 ? (uu & (heads - 1)) : uu - lr * heads;
      row[t] = cx.row0 + lr;
      int fi = fi0 + lr, sq = sq0;
      while (fi >= N) { fi -= N; ++sq; }
      const float* base = p.QKVacc + static_cast<size_t>(sq) * N * ld + hh[t] * hd + lane * VPL;
      j0[t] = max(0, fi - win);
      const int j1 = min(N - 1, fi + win);
      nk[t] = j1 - j0[t] + 1;
      F32Vec<VPL>::ld(base + static_cast<size_t>(fi) * ld, q[t]);
#pragma unroll
      for (int k = 0; k < KB; ++k) {
        const int j = min(j0[t] + k, j1);
        F32Vec<VPL>::ld(base + static_cast<size_t>(j) * ld + H, kv[t][k]);
        F32Vec<VPL>::ld(base + static_cast<size_t>(j) * ld + 2 * H, vv[t][k]);
      }
    }
#pragma unroll
    for (int t = 0; t < U; ++t) {
      const float* bq = bqkv + hh[t] * hd + lane * VPL;
      float s[KB];
#pragma unroll
      for (int k = 0; k < VPL; ++k) q[t][k] += __ldg(bq + k);
#pragma unroll
      for (int c = 0; c < KB; ++c) {
        float d = 0.f;
#pragma unroll
        for (int k = 0; k < VPL; ++k) d = fmaf(q[t][k], kv[t][c][k] + __ldg(bq + H + k), d);
        s[c] = d;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int c = 0; c < KB; ++c) s[c] += __shfl_xor_sync(0xffffffffu, s[c], o);
      float mx = -INFINITY;
#pragma unroll
      for (int c = 0; c < KB; ++c) { s[c] = c < nk[t] ? s[c] * scale : -INFINITY; mx = fmaxf(mx, s[c]); }
      float den = 0.f, acc[VPL];
#pragma unroll
      for (int k = 0; k < VPL; ++k) acc[k] = 0.f;
#pragma unroll
      for (int c = 0; c < KB; ++c) {
        const float pr = __expf(s[c] - mx);          // exp(-inf) = 0 for the masked slots
        den += pr;
#pragma unroll
        for (int k = 0; k < VPL; ++k) acc[k] = fmaf(pr, vv[t][c][k], acc[k]);
      }
      if (valid[t]) {
        const float inv = __fdividef(1.f, den);
        __nv_bfloat16* op = cx.A2 + win_tiled_off(row[t] - cx.row0, hh[t] * hd + lane * VPL, cx.RgP);   // VPL <= 4 elements stay inside one 16-byte chunk
        float o[VPL];
#pragma unroll
        for (int k = 0; k < VPL; ++k) o[k] = fmaf(acc[k], inv, __ldg(bq + 2 * H + k));   // sum_c p_c (v_c + b) / den = sum_c p_c v_c / den + b
        if constexpr (VPL == 4) {
          *reinterpret_cast<uint2*>(op) = f32x4_to_bf16(o);
        } else {
#pragma unroll
          for (int k = 0; k < VPL; ++k) op[k] = __float2bfloat16_rn(o[k]);
        }
      }
    }
  }
}

// General band width: one unit per warp, keys in batches of 4 with an online softmax (compact code; rarely used).
template <int VPL>
__device__ __forceinline__ void win_attn_wide(const WinParams& p, const WinCtx& cx, const float* __restrict__ bqkv) {
  const int lane = threadIdx.x & 31, mw = (threadIdx.x >> 5) - 1;
  constexpr int hd = VPL * 32, KB = 4;
  const int N = p.s.N, heads = p.heads, H = p.s.H, ld = 3 * H;
  const int n_units = cx.nrows * heads;
  const float scale = rsqrtf(static_cast<float>(hd));
  const int win = p.window;
#pragma unroll 1
  for (int u = cx.rank + cx.nranks * mw; u < n_units; u += cx.nranks * 8) {
    const int h = u % heads, row = cx.row0 + u / heads, fi = row % N, sq = row / N;
    const float* base = p.QKVacc + static_cast<size_t>(sq) * N * ld + h * hd + lane * VPL;
    const float* bq = bqkv + h * hd + lane * VPL;
    float q[VPL], bk[VPL];
    F32Vec<VPL>::ld(base + static_cast<size_t>(fi) * ld, q);
#pragma unroll
    for (int k = 0; k < VPL; ++k) { q[k] += __ldg(bq + k); bk[k] = __ldg(bq + H + k); }
    const int j0 = max(0, fi - win), j1 = min(N - 1, fi + win);
    float mx = -INFINITY, den = 0.f, acc[VPL];
#pragma unroll
    for (int k = 0; k < VPL; ++k) acc[k] = 0.f;
#pragma unroll 1
    for (int jb = j0; jb <= j1; jb += KB) {
      float kv[KB][VPL], vv[KB][VPL], s[KB];
#pragma unroll
      for (int c = 0; c < KB; ++c) {
        const int j = min(jb + c, j1);
        F32Vec<VPL>::ld(base + static_cast<size_t>(j) * ld + H, kv[c]);
        F32Vec<VPL>::ld(base + static_cast<size_t>(j) * ld + 2 * H, vv[c]);
      }
#pragma unroll
      for (int c = 0; c < KB; ++c) {
        float d = 0.f;
#pragma unroll
        for (int k = 0; k < VPL; ++k) d = fmaf(q[k], kv[c][k] + bk[k], d);
        s[c] = d;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int c = 0; c < KB; ++c) s[c] += __shfl_xor_sync(0xffffffffu, s[c], o);
#pragma unroll
      for (int c = 0; c < KB; ++c) {
        if (jb + c <= j1) {
          const float sc = s[c] * scale;
          const float nmx = fmaxf(mx, sc);
          const float corr = __expf(mx - nmx), pr = __expf(sc - nmx);
          den = den * corr + pr;
#pragma unroll
          for (int k = 0; k < VPL; ++k) acc[k] = fmaf(acc[k], corr, pr * vv[c][k]);
          mx = nmx;
        }
      }
    }
    const float inv = __fdividef(1.f, den);
    __nv_bfloat16* op = cx.A2 + win_tiled_off(row - cx.row0, h * hd + lane * VPL, cx.RgP);
#pragma unroll
    for (int k = 0; k < VPL; ++k) op[k] = __float2bfloat16_rn(fmaf(acc[k], inv, __ldg(bq + 2 * H + k)));
  }
}

// GELU stage: Hm = bf16( GELU_tanh(Hacc + b_fc1) ), Hacc <- 0      (timm Mlp: fc1 -> act, FMT.py:159-162)
__device__ __forceinline__ float gelu_tanh_fast(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  const float u = k0 * (x + k1 * x * x * x);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  return 0.5f * x * (1.0f + t);
}
__device__ __forceinline__ void win_gelu_stage(const WinParams& p, const WinCtx& cx, const float* __restrict__ b1, unsigned epoch) {
  const int M4 = p.mlp_hidden;
  const unsigned total4 = static_cast<unsigned>(cx.nrows) * M4 / 4;      // this group's elements; i = local float4 index
  const unsigned stride = cx.nranks * WIN_MAIN;
  float* hacc = p.Hacc + static_cast<size_t>(cx.row0) * M4;
  constexpr int NB = 6;                                  // float4 per thread per batch (R = 180, 4096 hidden: 5 per thread)
  for (unsigned i0 = cx.rank * WIN_MAIN + (threadIdx.x - 32); i0 < total4; i0 += NB * stride) {
    float4 a[NB], b[NB];
    win_mark(p, epoch, 0);
#pragma unroll
    for (int k = 0; k < NB; ++k) {
      const unsigned i = i0 + k * stride;
      if (i < total4) {
        a[k] = ldcg4(hacc + static_cast<size_t>(i) * 4);
        b[k] = __ldg(reinterpret_cast<const float4*>(b1 + (i * 4) % static_cast<unsigned>(M4)));
      }
    }
#pragma unroll
    for (int k = 0; k < NB; ++k) {
      const unsigned i = i0 + k * stride;
      if (i < total4) {
        if (k == 0) win_mark(p, epoch, 1);
        float v[4] = {gelu_tanh_fast(a[k].x + b[k].x), gelu_tanh_fast(a[k].y + b[k].y), gelu_tanh_fast(a[k].z + b[k].z), gelu_tanh_fast(a[k].w + b[k].w)};
        {
          const unsigned e4 = i * 4, M4u = static_cast<unsigned>(M4);
          *reinterpret_cast<uint2*>(cx.Hm + win_tiled_off(static_cast<int>(e4 / M4u), static_cast<int>(e4 % M4u), cx.RgP)) = f32x4_to_bf16(v);
        }
        *reinterpret_cast<float4*>(hacc + static_cast<size_t>(i) * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    win_mark(p, epoch, 2);
  }
  win_mark(p, epoch, 3);
}

// COMB stage: decoder bias, CFG combine (FMT.py:375-379,396-399), then the explicit Runge-Kutta bookkeeping of stage g of
// step `step` (Euler: y += dt * v).  Writes the x-embedder operand `ax` of the next evaluation and zeroes Vacc.
__device__ __forceinline__ void win_comb_stage(const WinParams& p, const WinCtx& cx, int step, int g) {
  const ModelShape& s = p.s;
  const int G = p.n_stages;
  const size_t per_branch = static_cast<size_t>(s.B) * s.N * s.W;
  const size_t nx = static_cast<size_t>(s.B) * s.L * s.W;
  for (unsigned i = cx.all_rank * WIN_MAIN + (threadIdx.x - 32); i < per_branch; i += cx.all_n * WIN_MAIN) {   // R <= 256 rows: 32-bit indices
    const int j = static_cast<int>(i % static_cast<unsigned>(s.W));
    const int f = static_cast<int>((i / static_cast<unsigned>(s.W)) % static_cast<unsigned>(s.N)), b = static_cast<int>(i / static_cast<unsigned>(s.W * s.N));
    const bool cur = f >= s.P;
    const size_t o = cur ? (static_cast<size_t>(b) * s.L + (f - s.P)) * s.W + j : 0;
    // ---- every load of this element first
    float vb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int br = 0; br < 4; ++br)
      if (br < s.nb) vb[br] = __ldcg(p.Vacc + br * per_branch + i);
    const float bd = __ldg(p.b_dec + j);
    const float dt = __ldg(p.ddt + step);
    const SlotArgs* const slots = p.wargs->slots;
    float a_s, r_s, e_s;
    int nb;
    const float y0 = cur ? __ldcg(p.x_state + o) : 0.f;
    float kprev[4] = {0.f, 0.f, 0.f, 0.f};
    if (G > 1 && cur) {
#pragma unroll
      for (int jj = 0; jj < 3; ++jj)
        if (jj < g) kprev[jj] = __ldcg(p.kbuf + static_cast<size_t>(jj) * nx + o);
    }
    // ---- then the arithmetic and the stores
#pragma unroll
    for (int br = 0; br < 4; ++br)
      if (br < s.nb) { vb[br] += bd; p.Vacc[br * per_branch + i] = 0.f; }
    if (!cur) continue;
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
      const float* c = last ? p.rk_b : &p.rk_a[(g + 1) * G];
      float acc = 0.f;
#pragma unroll
      for (int jj = 0; jj < 4; ++jj)
        if (jj <= g && c[jj] != 0.f) acc = fmaf(c[jj], jj == g ? v : kprev[jj], acc);
      y = fmaf(dt, acc, y0);
      if (last) p.x_state[o] = y;
    }
    const __nv_bfloat16 t = __float2bfloat16_rn(y);
    for (int br = 0; br < s.nb; ++br) p.ax[((static_cast<size_t>(br) * s.B + b) * s.N + f) * s.W + j] = t;
  }
}

__device__ __forceinline__ void win_attn_dispatch(const WinParams& p, const WinCtx& cx, const float* bqkv) {
  const int hd = p.s.H / p.heads;
  if (p.window <= 2) {
    if (hd == 128) win_attn_band5<4, 2>(p, cx, bqkv);
    else if (hd == 64) win_attn_band5<2, 2>(p, cx, bqkv);
    else win_attn_band5<1, 2>(p, cx, bqkv);
  } else {
    if (hd == 128) win_attn_wide<4>(p, cx, bqkv);
    else if (hd == 64) win_attn_wide<2>(p, cx, bqkv);
    else win_attn_wide<1>(p, cx, bqkv);
  }
}

// ---------------------------------------------------------------------------------------------------------------- kernel
// This CTA's rows, rank and operand buffers in the SIMT stages (one thread writes them)
template <bool GROUPED>
__device__ __forceinline__ void win_ctx(const WinParams& p, WinCtx& cx) {
  if (GROUPED) {
    const int g = blockIdx.x / p.Cg;
    const size_t t_a1 = static_cast<size_t>((p.s.H + 63) / 64) * p.RgP * 64, t_hm = static_cast<size_t>((p.mlp_hidden + 63) / 64) * p.RgP * 64;
    cx.row0 = g * p.Rg; cx.nrows = p.Rg; cx.rank = blockIdx.x % p.Cg; cx.nranks = p.Cg;
    cx.all_rank = blockIdx.x; cx.all_n = p.G * p.Cg; cx.RgP = p.RgP;
    cx.A1 = p.A1 + g * t_a1; cx.A2 = p.A2 + g * t_a1; cx.Hm = p.Hm + g * t_hm;
    cx.bar = p.bar_counter + 32 * (1 + g);
  } else {
    cx.row0 = 0; cx.nrows = p.R; cx.rank = blockIdx.x; cx.nranks = gridDim.x; cx.all_rank = blockIdx.x; cx.all_n = gridDim.x; cx.RgP = p.Rp;
    cx.A1 = p.A1; cx.A2 = p.A2; cx.Hm = p.Hm; cx.bar = p.bar_counter;
  }
}

template <int NV /* dim_h / 128 */, bool GROUPED /* false: split-K over the whole grid; true: one group of CTAs per <= 128 rows */>
__global__ void __launch_bounds__(WIN_THREADS, 1) fmt_window_kernel(const WinParams* __restrict__ pp) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ WinParams p;
  __shared__ float red_smem[16];
  __shared__ WinItems items;
  __shared__ unsigned bar_ctr[4];                // barriers passed: [0] total (trace index), [1] on the group counter, [2] on the grid counter
  __shared__ WinRing rings[WIN_THREADS / 32];   // ring positions of each role warp live here between GEMM stages (registers are scarce: 168 at 288 threads)
  __shared__ WinCtx cx;                  // shared, not local: a stack object is re-fetched from L2 after every grid barrier (the acquire invalidates L1)
  {
    const int4* src = reinterpret_cast<const int4*>(pp);
    int4* dst = reinterpret_cast<int4*>(&p);
    for (int i = threadIdx.x; i < static_cast<int>(sizeof(WinParams) / 16); i += WIN_THREADS) dst[i] = src[i];
  }
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  WinSmem sm;
  sm.nw = GROUPED ? WIN2_NW : WIN_NW;
  sm.w_bytes = GROUPED ? WIN2_W_BYTES : WIN_W_BYTES;
  sm.wring = smem;
  sm.aring = smem + sm.nw * sm.w_bytes;
  sm.stg = reinterpret_cast<float*>(sm.aring + (GROUPED ? WIN2_A_RING : WIN_A_RING));     // staging exists in the split-K schedule only
  sm.w_full = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sm.stg) + (GROUPED ? 0 : 2 * WIN_STG_BYTES));
  sm.w_empty = sm.w_full + WIN_MAX_NA;
  sm.a_full = sm.w_empty + WIN_MAX_NA;
  sm.a_empty = sm.a_full + WIN_MAX_NA;
  sm.t_full = sm.a_empty + WIN_MAX_NA;
  sm.tmem_slot = reinterpret_cast<uint32_t*>(sm.t_full + 1);
  sm.gate = reinterpret_cast<int*>(sm.tmem_slot + 1);
  __syncthreads();
  if (GROUPED && static_cast<int>(blockIdx.x) >= p.G * p.Cg) return;    // CTAs left over by 148 = G * Cg + rest have no work

  if (threadIdx.x == 0) win_ctx<GROUPED>(p, cx);
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int g = threadIdx.x; g < p.n_gemms; g += WIN_THREADS) {
    int nt, kb0, kb1;
    const bool has = GROUPED ? win_item2(p.gemms[g], cx, nt, kb0, kb1) : win_item(p.gemms[g], nt, kb0, kb1);
    items.it[g] = make_int4(has ? nt : -1, kb0, kb1, 0);
  }
  int NA = GROUPED ? WIN2_NA : WIN_A_RING / (cx.RgP * 128);
  if (NA > WIN_MAX_NA) NA = WIN_MAX_NA;
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < sm.nw; ++i) { mbar_init(&sm.w_full[i], 1); mbar_init(&sm.w_empty[i], 1); }
    for (int i = 0; i < WIN_MAX_NA; ++i) { mbar_init(&sm.a_full[i], 1); mbar_init(&sm.a_empty[i], 1); }
    mbar_init(sm.t_full, 1);
    *sm.gate = 0;
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(sm.tmem_slot, 256);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *sm.tmem_slot;
  const int n_eval = p.n_steps * p.n_stages;

  if (warp == 0) {
    if (lane == 0) {
      if (GROUPED) win_weight_producer2(p, items, sm, n_eval);
      else win_weight_producer(p, items, sm, n_eval);
    }
    __syncwarp();
  } else {
    // One call site per stage kind: the stage list of an evaluation is decoded from its index, so the GEMM stage (ring
    // state in registers) is inlined exactly once and the hot code stays small.  With bs = 8 stages per block:
    //   0: x_embedder GEMM   1: ROW (init)   2 + bs*blk + {0: qkv GEMM, 1: ATTN, 2: proj GEMM, 3: ROW, 4: fc1 GEMM, 5: GELU,
    //   6: fc2 GEMM, 7: ROW}   spe-2: decoder GEMM   spe-1: COMB
    // (grouped schedule with the GELU fused into fc1's epilogue: bs = 7, {..., 4: fc1 GEMM + GELU, 5: fc2 GEMM, 6: ROW})
    if (lane == 0) rings[warp] = WinRing();
    __syncwarp();
    if (threadIdx.x == 32) { bar_ctr[0] = 0; bar_ctr[1] = 0; bar_ctr[2] = 0; bar_ctr[3] = 0; }
    named_bar_sync(1, WIN_MAIN);
    volatile unsigned* ctr = bar_ctr;
    // Loop invariants are re-read from shared memory (volatile) where they are used instead of living in registers across the
    // stages: the kernel has exactly as many registers as it needs, and a spilled value costs an L2 round trip per barrier.
    const volatile WinParams& pv = p;
    const int bs = (GROUPED && pv.fuse_gelu) ? 7 : 8;
    while (static_cast<int>(ctr[3]) < pv.n_steps * pv.n_stages) {
      for (int si = 0; si < 4 + bs * pv.depth; ++si) {
        const int e = static_cast<int>(ctr[3]);
        const int D = pv.depth, spe = 4 + bs * D;
        const long long H = pv.s.H;
        const __nv_bfloat16* table_e = p.table + static_cast<size_t>(e) * (static_cast<size_t>(pv.R) * pv.NT);
        const bool is_edge = si < 2 || si >= spe - 2;
        // block and position inside it (8-stage numbering); divisions by the CONSTANTS 8 and 7 only (shift / multiply-shift)
        const int blk = is_edge ? 0 : (bs == 8 ? (si - 2) >> 3 : (si - 2) / 7);
        int j = is_edge ? 0 : (bs == 8 ? (si - 2) & 7 : (si - 2) % 7);
        if (bs == 7 && j >= 5) ++j;
        const bool is_gemm = is_edge ? (si == 0 || si == spe - 2) : ((j & 1) == 0);
        if (is_gemm) {
          const int g = si == 0 ? 0 : (si == spe - 2 ? 1 + 4 * D : 1 + 4 * blk + (j >> 1));
          WinRing rg = rings[warp];
          if (GROUPED) win_gemm2_stage(p, cx, p.gemms[g], items.it[g], sm, rg, tmem_base, ctr[0], (!is_edge && j == 4) ? p.b_fc1[blk] : nullptr);
          else win_gemm_stage(p, p.gemms[g], items.it[g], sm, rg, NA, tmem_base, ctr[0]);
          __syncwarp();                      // every lane has read rings[warp] before lane 0 overwrites it
          if (lane == 0) rings[warp] = rg;
          __syncwarp();
        } else {
          if (si == spe - 1) {
            win_comb_stage(p, cx, e / p.n_stages, e % p.n_stages);
          } else if (si == 1) {
            win_row_stage<NV>(p, cx, red_smem, table_e, 0, p.b_x, 0, 0, H, false);      // LN + modulate with block 0's (shift_msa, scale_msa)
          } else if (j == 1) {
            win_attn_dispatch(p, cx, p.b_qkv[blk]);
          } else if (j == 5) {
            win_gelu_stage(p, cx, p.b_fc1[blk], ctr[0]);
          } else {
            const long long base = static_cast<long long>(blk) * 6 * H;
            // j == 3: after proj -> gate_msa, then the mlp modulation; j == 7: after fc2 -> gate_mlp, then the NEXT block's msa
            // modulation or, after the last block, the decoder's (shift, scale)
            const bool after_proj = (j == 3);
            const long long gate_off = base + (after_proj ? 2 : 5) * H;
            const long long mod = after_proj ? base + 3 * H : base + 6 * H;
            win_row_stage<NV>(p, cx, red_smem, table_e, 1, after_proj ? p.b_proj[blk] : p.b_fc2[blk], gate_off, mod, mod + H, after_proj);
          }
          if (threadIdx.x == 32) atomicAdd(sm.gate, 1);                             // quiet point of a SIMT stage: its loads have landed
        }
        // The CFG combine reads every branch, and the next x-embedder GEMM reads what it wrote: the barriers around COMB span
        // the whole grid; every other stage only depends on rows of its own group.
        if (!GROUPED || si >= spe - 2) win_grid_sync(p, ctr, p.bar_counter, 2, cx.all_n, si == spe - 1);
        else win_grid_sync(p, ctr, cx.bar, 1, cx.nranks, false);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 256);
}

}  // namespace fmt
