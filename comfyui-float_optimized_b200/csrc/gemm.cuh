// GEMMs of the FMT step:  out[M,N] = epilogue( A[M,K] . W[N,K]^T )
//   * gemm_tc_kernel   - bf16 operands, tcgen05.mma (cta_group::1, M=128 x N=BN x K=16) with fp32 accumulators in
//                        TMEM, operands staged by TMA (128B swizzle) through an mbarrier ring; persistent over
//                        output tiles with a double-buffered accumulator so the epilogue of tile i overlaps the
//                        MMAs of tile i+1.  Warp roles: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 4..11 = epilogue.
//                        SPLIT = true (FMT_MODE_BF16X3): bf16 hi / lo operand pairs (bf16x3_t below), three MMAs per K step
//                        (Ah.Wh + Ah.Wl + Al.Wh) into the same accumulator; fp32-class products on the tensor pipe.
//   * gemm_tc2_kernel  - the same on CTA pairs (cta_group::2), same SPLIT variant.
//   * gemm_simt_kernel - fp32 operands, plain FFMA tiles; FMT_MODE_FP32_VALIDATE only (the 1e-4 parity mode).
// Both share epi_apply(), which carries the fused epilogues of the reference's block
// (FMT.py:171-176): bias, GELU(tanh), +pos_embed, and x += gate * (.).
#pragma once
#include <type_traits>
#include "ptx.cuh"

namespace fmt {

enum EpiKind : int { EPI_STORE = 0, EPI_GELU = 1, EPI_POS = 2, EPI_GATE_RES = 3 };

struct EpiParams {
  int kind;
  int M, N;
  const float* bias;   // [N] or nullptr
  void* out;           // [M, ldo]: float if out_f32 else the activation type AT
  int ldo;
  int out_f32;
  const float* pos;    // EPI_POS: out += pos[(m % frames) * N + n]
  int frames;
  const void* gate;    // EPI_GATE_RES: table (type TT), element (urow[m] * ldg + gate_off + n)
  const int* urow;     // row indirection into the table (nullptr = identity)
  long long ldg;
  long long gate_off;
  int raster_gm;       // CTA-pair kernel: row-tiles per raster group (>= 1)
  int ksplit;          // CTA-pair kernel, EPI_GATE_RES only: K slices per tile (0/1 = none); partial sums meet in x through fp32 RED
};

__device__ __forceinline__ float gelu_tanh(float x) {
  // nn.GELU(approximate="tanh"), FMT.py:161
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  float u = k0 * (x + k1 * x * x * x);
  return 0.5f * x * (1.0f + tanhf(u));
}

__device__ __forceinline__ float gelu_tanh_approx(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  const float u = k0 * (x + k1 * x * x * x);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  return 0.5f * x * (1.0f + t);
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

// 256-bit global store (sm_100+): one full 32-byte L2 sector per lane.  The tcgen05 epilogues hold one output ROW per lane,
// so a warp-wide store instruction touches 32 different lines; with 16-byte stores every sector was written in two halves
// (partial-sector writes -> L2 fill reads from DRAM and ~3x longer epilogues), with 32-byte stores each sector is written once.
__device__ __forceinline__ void st_global_v8(void* p, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t a4, uint32_t a5, uint32_t a6,
                                             uint32_t a7) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(a4), "r"(a5), "r"(a6),
               "r"(a7)
               : "memory");
}
__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// row segment of 32 values per lane -> global, in 32-byte pieces
__device__ __forceinline__ void store_row32(float* p, const float (&v)[32]) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
    st_global_v8(p + 8 * i, __float_as_uint(v[8 * i]), __float_as_uint(v[8 * i + 1]), __float_as_uint(v[8 * i + 2]), __float_as_uint(v[8 * i + 3]),
                 __float_as_uint(v[8 * i + 4]), __float_as_uint(v[8 * i + 5]), __float_as_uint(v[8 * i + 6]), __float_as_uint(v[8 * i + 7]));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ void store_row32(__nv_bfloat16* p, const float (&v)[32]) {
#pragma unroll
  for (int i = 0; i < 2; ++i)
    st_global_v8(p + 16 * i, pack_bf16x2(v[16 * i], v[16 * i + 1]), pack_bf16x2(v[16 * i + 2], v[16 * i + 3]), pack_bf16x2(v[16 * i + 4], v[16 * i + 5]),
                 pack_bf16x2(v[16 * i + 6], v[16 * i + 7]), pack_bf16x2(v[16 * i + 8], v[16 * i + 9]), pack_bf16x2(v[16 * i + 10], v[16 * i + 11]),
                 pack_bf16x2(v[16 * i + 12], v[16 * i + 13]), pack_bf16x2(v[16 * i + 14], v[16 * i + 15]));
}

// bf16x3 operands (FMT_MODE_BF16X3): x = hi + lo with hi = bf16(x) and lo = bf16(x - hi); the split GEMM sums Ah.Wh + Ah.Wl + Al.Wh
// (Al.Wl, ~2^-16 relative, is dropped).  A pair matrix has rows of 2K bf16 values in which every 64-column K block of hi is followed by
// the same block of lo: [hi 0:64 | lo 0:64 | hi 64:128 | lo 64:128 | ...], so one tensor map per operand serves both halves (box
// columns 128 kb and 128 kb + 64).  bf16x3_t stands for one element of such a row and is 4 bytes, so a pair row takes the bytes of
// an fp32 row of the same K and kernels index a pair matrix like any other (p = base + row * ld + c).  Buffers are 256-byte aligned
// and ld is a multiple of 64, so the byte offset of p names the element's 64-column block (offset / 256) and its column c % 64
// in the block (offset % 256 / 4): split_hi(p) is where its hi part really is, its lo part sits 64 values (128 bytes) further.
struct bf16x3_t { uint32_t bits; };
__device__ __forceinline__ __nv_bfloat16* split_hi(bf16x3_t* p) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  return reinterpret_cast<__nv_bfloat16*>((a & ~static_cast<uintptr_t>(255)) + ((a & 255) >> 1));
}
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  const __nv_bfloat162 l = __floats2bfloat162_rn(a - __low2float(h), b - __high2float(h));
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

template <typename T, int NC> struct VecIO;
template <int NC> struct VecIO<float, NC> {
  static_assert(NC % 4 == 0, "");
  static __device__ __forceinline__ void load(const float* p, float (&v)[NC]) {
#pragma unroll
    for (int i = 0; i < NC / 4; ++i) {
      float4 t = reinterpret_cast<const float4*>(p)[i];
      v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
    }
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[NC]) {
#pragma unroll
    for (int i = 0; i < NC / 4; ++i) reinterpret_cast<float4*>(p)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
  }
};
template <int NC> struct VecIO<__nv_bfloat16, NC> {
  static_assert(NC % 4 == 0, "");
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[NC]) {
#pragma unroll
    for (int i = 0; i < NC / 4; ++i) {
      uint2 t = reinterpret_cast<const uint2*>(p)[i];
      __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&t.x), b = *reinterpret_cast<__nv_bfloat162*>(&t.y);
      v[4 * i] = __low2float(a); v[4 * i + 1] = __high2float(a); v[4 * i + 2] = __low2float(b); v[4 * i + 3] = __high2float(b);
    }
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[NC]) {
#pragma unroll
    for (int i = 0; i < NC / 4; ++i) {
      __nv_bfloat162 a = __floats2bfloat162_rn(v[4 * i], v[4 * i + 1]), b = __floats2bfloat162_rn(v[4 * i + 2], v[4 * i + 3]);
      uint2 t;
      t.x = *reinterpret_cast<uint32_t*>(&a);
      t.y = *reinterpret_cast<uint32_t*>(&b);
      reinterpret_cast<uint2*>(p)[i] = t;
    }
  }
};

// NC consecutive elements starting at a multiple of NC (NC divides 64: one K block): NC hi values, then NC lo values 128 bytes further
template <int NC> struct VecIO<bf16x3_t, NC> {
  static_assert(NC % 4 == 0 && 64 % NC == 0, "");
  static __device__ __forceinline__ void store(bf16x3_t* p, const float (&v)[NC]) {
    uint32_t hi[NC / 2], lo[NC / 2];
#pragma unroll
    for (int i = 0; i < NC / 2; ++i) split_bf16x2(v[2 * i], v[2 * i + 1], hi[i], lo[i]);
    __nv_bfloat16* hp = split_hi(p);
    if constexpr (NC % 16 == 0) {
#pragma unroll
      for (int i = 0; i < NC / 16; ++i) {
        st_global_v8(hp + 16 * i, hi[8 * i], hi[8 * i + 1], hi[8 * i + 2], hi[8 * i + 3], hi[8 * i + 4], hi[8 * i + 5], hi[8 * i + 6], hi[8 * i + 7]);
        st_global_v8(hp + 64 + 16 * i, lo[8 * i], lo[8 * i + 1], lo[8 * i + 2], lo[8 * i + 3], lo[8 * i + 4], lo[8 * i + 5], lo[8 * i + 6], lo[8 * i + 7]);
      }
    } else {
#pragma unroll
      for (int i = 0; i < NC / 4; ++i) {
        reinterpret_cast<uint2*>(hp)[i] = make_uint2(hi[2 * i], hi[2 * i + 1]);
        reinterpret_cast<uint2*>(hp + 64)[i] = make_uint2(lo[2 * i], lo[2 * i + 1]);
      }
    }
  }
};

// One thread owns NC consecutive columns [n0, n0+NC) of row m (n0 % NC == 0, N % NC == 0).
template <typename AT, typename TT, int NC>
__device__ __forceinline__ void epi_apply(const EpiParams& p, int m, int n0, float (&v)[NC]) {
  if (p.bias != nullptr) {
    float b[NC];
    VecIO<float, NC>::load(p.bias + n0, b);
#pragma unroll
    for (int i = 0; i < NC; ++i) v[i] += b[i];
  }
  if (p.kind == EPI_GELU) {
#pragma unroll
    for (int i = 0; i < NC; ++i) v[i] = sizeof(AT) == 2 ? gelu_tanh_approx(v[i]) : gelu_tanh(v[i]);   // bf16 output: tanh.approx (2^-11) is below its rounding
  } else if (p.kind == EPI_POS) {
    float b[NC];
    VecIO<float, NC>::load(p.pos + static_cast<size_t>(m % p.frames) * p.N + n0, b);
#pragma unroll
    for (int i = 0; i < NC; ++i) v[i] += b[i];
  } else if (p.kind == EPI_GATE_RES) {
    const int ur = p.urow ? p.urow[m] : m;
    float g[NC], x[NC];
    VecIO<TT, NC>::load(reinterpret_cast<const TT*>(p.gate) + static_cast<size_t>(ur) * p.ldg + p.gate_off + n0, g);
    float* xp = reinterpret_cast<float*>(p.out) + static_cast<size_t>(m) * p.ldo + n0;
    VecIO<float, NC>::load(xp, x);
#pragma unroll
    for (int i = 0; i < NC; ++i) x[i] = fmaf(g[i], v[i], x[i]);     // x = x + gate * branch  (FMT.py:174-175)
    if constexpr (NC == 32) store_row32(xp, x);
    else VecIO<float, NC>::store(xp, x);
    return;
  }
  if (p.out_f32) {
    float* op = reinterpret_cast<float*>(p.out) + static_cast<size_t>(m) * p.ldo + n0;
    if constexpr (NC == 32) store_row32(op, v);
    else VecIO<float, NC>::store(op, v);
  } else {
    AT* op = reinterpret_cast<AT*>(p.out) + static_cast<size_t>(m) * p.ldo + n0;
    if constexpr (NC == 32 && sizeof(AT) == 2) store_row32(reinterpret_cast<__nv_bfloat16*>(op), v);
    else VecIO<AT, NC>::store(op, v);
  }
}

// ------------------------------------------------------------------------------------------------
// tcgen05 / TMA GEMM
// ------------------------------------------------------------------------------------------------
template <int BN, bool SPLIT = false> struct TcCfg {
  static constexpr int BM = 128, BK = 64, UMMA_K = 16;
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int HALVES = SPLIT ? 2 : 1;           // SPLIT: a stage holds [Ah | Wh | Al | Wl] of one K block
  static constexpr int STAGE_BYTES = HALVES * (A_BYTES + B_BYTES);
  static constexpr int STAGES = SPLIT ? ((BN == 256) ? 2 : (BN == 128 ? 3 : 4)) : ((BN == 256) ? 4 : (BN == 128 ? 6 : 8));
  static constexpr int ACC_STAGES = 2;
  static constexpr int TMEM_COLS = ACC_STAGES * BN;     // 128 / 256 / 512: powers of two >= 32
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + BAR_BYTES + 1024;   // +1024: manual 1 KB alignment for SWIZZLE_128B
  static constexpr int EPI_WARPS = 8;                    // warps 4..11: two per TMEM lane quarter, each takes every other 32-column chunk
  static constexpr int THREADS = 128 + EPI_WARPS * 32;   // warpgroup 0 = TMA producer, MMA issuer, TMEM allocator, one idle warp
  static_assert(BN == 64 || BN == 128 || BN == 256, "BN");
};

// SPLIT: tmA / tmB describe pair matrices (2K bf16 columns), K is the logical depth; activation outputs are bf16x3_t pairs.
template <int BN, typename TT, bool SPLIT>
__global__ void __launch_bounds__(TcCfg<BN, SPLIT>::THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const EpiParams ep, const int K) {
  using C = TcCfg<BN, SPLIT>;
  using AT = typename std::conditional<SPLIT, bf16x3_t, __nv_bfloat16>::type;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tfull_bar = empty_bar + C::STAGES;
  uint64_t* tempty_bar = tfull_bar + C::ACC_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + C::ACC_STAGES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_kb = (K + C::BK - 1) / C::BK;
  const int m_tiles = (ep.M + C::BM - 1) / C::BM;
  const int n_tiles = (ep.N + BN - 1) / BN;
  const int total_tiles = m_tiles * n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < C::STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < C::ACC_STAGES; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], C::EPI_WARPS); }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, C::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();

  // register budget per warpgroup: the role warps need few registers, the fused epilogues many (residual + gate rows in flight).
  // The setmaxnreg sits INSIDE each role branch: ptxas budgets a region that both branches reach with the smaller value.
  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      pdl_wait_prior_grid();
      int stage = 0; uint32_t phase = 0;
      for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        const int m0 = (t % m_tiles) * C::BM, n0 = (t / m_tiles) * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * C::STAGE_BYTES;
          mbar_expect_tx(&full_bar[stage], C::STAGE_BYTES);
          tma_load_2d(&tmA, &full_bar[stage], sa, kb * C::BK * C::HALVES, m0, kEvictNormal);
          tma_load_2d(&tmB, &full_bar[stage], sa + C::A_BYTES, kb * C::BK * C::HALVES, n0, kEvictNormal);
          if constexpr (SPLIT) {
            tma_load_2d(&tmA, &full_bar[stage], sa + C::A_BYTES + C::B_BYTES, kb * C::BK * 2 + C::BK, m0, kEvictNormal);
            tma_load_2d(&tmB, &full_bar[stage], sa + 2 * C::A_BYTES + C::B_BYTES, kb * C::BK * 2 + C::BK, n0, kEvictNormal);
          }
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_bf16_f32(C::BM, BN);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);        // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);              // TMA bytes have landed
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * C::STAGE_BYTES);
          const uint64_t da = make_sw128_kmajor_desc(sa);
          const uint64_t db = make_sw128_kmajor_desc(sa + C::A_BYTES);
#pragma unroll
          for (int k = 0; k < C::BK / C::UMMA_K; ++k) {
            // advance along K inside the 128B swizzle atom: +32 bytes (>>4 = 2) per UMMA_K
            umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
          }
          if constexpr (SPLIT) {                           // the lo products of the same K block: Ah.Wl + Al.Wh
            const uint64_t dal = make_sw128_kmajor_desc(sa + C::A_BYTES + C::B_BYTES), dbl = make_sw128_kmajor_desc(sa + 2 * C::A_BYTES + C::B_BYTES);
#pragma unroll
            for (int k = 0; k < C::BK / C::UMMA_K; ++k) {
              umma_bf16(d_tmem, da + 2 * k, dbl + 2 * k, idesc, 1u);
              umma_bf16(d_tmem, dal + 2 * k, db + 2 * k, idesc, 1u);
            }
          }
          umma_commit(&empty_bar[stage]);                  // frees the smem slot when these MMAs retire
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull_bar[acc]);                      // accumulator complete -> epilogue
        if (++acc == C::ACC_STAGES) { acc = 0; acc_phase ^= 1; }
      }
    }
    __syncwarp();
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
    // ===================== epilogue warps (TMEM -> registers -> global) =====================
    // Eight warps: with the fused epilogues (GELU, gate + residual) four warps - one per scheduler - took longer over a tile than
    // the tensor pipe over its main loop, and the GEMM ran at the epilogue's pace (fc1 at 32 clips: 63 us in the step against
    // 41 us with a plain store).  Two warps per lane quarter split the tile's column chunks.
    const int quarter = warp & 3;                          // a warp may only touch TMEM lanes [32*(warp%4), +32)
    const int half = (warp - 4) >> 2;                      // 0: even chunks, 1: odd chunks
    pdl_wait_prior_grid();
    int acc = 0; uint32_t acc_phase = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      const int m0 = (t % m_tiles) * C::BM, n0 = (t / m_tiles) * BN;
      const int m = m0 + quarter * 32 + lane;
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BN;
      if (ep.kind == EPI_GATE_RES) {
        // x += gate * (acc + bias), FMT.py:174-175.  The residual and gate rows of this warp's first chunk are requested BEFORE the
        // accumulator is waited for, those of its next chunk as soon as the current ones have been consumed: at K = 1024 a tile's
        // main loop lasts ~1 us, loading the rows inside the chunk loop made the epilogue twice as long as that (proj at 32 clips:
        // 22-33 us in the step against 17 us with a plain store).
        const bool row_ok = m < ep.M;
        const int mc = row_ok ? m : ep.M - 1;               // clamped row: loads stay in bounds, stores are predicated
        float* xrow = reinterpret_cast<float*>(ep.out) + static_cast<size_t>(mc) * ep.ldo + n0;
        const TT* grow = reinterpret_cast<const TT*>(ep.gate) + static_cast<size_t>(ep.urow ? ep.urow[mc] : mc) * ep.ldg + ep.gate_off + n0;
        const float* brow = ep.bias != nullptr ? ep.bias + n0 : nullptr;
        float4 xq[8], bq[8];
        constexpr int GW = 32 * sizeof(TT) / 16;            // 16-byte words per 32 gate values
        uint4 graw[GW];
        auto prefetch = [&](int c) {
          if (n0 + c * 32 < ep.N) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              xq[i] = *reinterpret_cast<const float4*>(xrow + c * 32 + i * 4);
              bq[i] = brow != nullptr ? __ldg(reinterpret_cast<const float4*>(brow + c * 32 + i * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int i = 0; i < GW; ++i) graw[i] = reinterpret_cast<const uint4*>(grow + c * 32)[i];
          }
        };
        prefetch(half);
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
#pragma unroll 1
        for (int c = half; c < BN / 32; c += 2) {
          float v[32], g[32];
          tmem_ld32(t_addr + c * 32, v);
          tmem_ld_wait();
          if constexpr (sizeof(TT) == 2) {
#pragma unroll
            for (int i = 0; i < GW; ++i) {
              const __nv_bfloat162* hp = reinterpret_cast<const __nv_bfloat162*>(&graw[i]);
#pragma unroll
              for (int k = 0; k < 4; ++k) { g[8 * i + 2 * k] = __low2float(hp[k]); g[8 * i + 2 * k + 1] = __high2float(hp[k]); }
            }
          } else {
#pragma unroll
            for (int i = 0; i < GW; ++i) { g[4 * i] = __uint_as_float(graw[i].x); g[4 * i + 1] = __uint_as_float(graw[i].y); g[4 * i + 2] = __uint_as_float(graw[i].z); g[4 * i + 3] = __uint_as_float(graw[i].w); }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            v[4 * i] = fmaf(g[4 * i], v[4 * i] + bq[i].x, xq[i].x);
            v[4 * i + 1] = fmaf(g[4 * i + 1], v[4 * i + 1] + bq[i].y, xq[i].y);
            v[4 * i + 2] = fmaf(g[4 * i + 2], v[4 * i + 2] + bq[i].z, xq[i].z);
            v[4 * i + 3] = fmaf(g[4 * i + 3], v[4 * i + 3] + bq[i].w, xq[i].w);
          }
          const bool ok = row_ok && n0 + c * 32 < ep.N;
          if (c + 2 < BN / 32) prefetch(c + 2);
          if (ok) store_row32(xrow + c * 32, v);
        }
      } else {
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
#pragma unroll 1
        for (int c = half; c < BN / 32; c += 2) {
          float v[32];
          tmem_ld32(t_addr + c * 32, v);
          tmem_ld_wait();
          const int n = n0 + c * 32;
          if (m < ep.M && n < ep.N) epi_apply<AT, TT, 32>(ep, m, n, v);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (++acc == C::ACC_STAGES) { acc = 0; acc_phase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, C::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------
// CTA-pair tcgen05 GEMM (cta_group::2): one 256 x BN output tile per pair of SMs.  Each CTA stages its own 128 rows of A
// and HALF of the B tile (BN/2 weight rows); the leader CTA issues M = 256 UMMAs that read both halves, so the shared-memory
// traffic per SM and per MMA drops from 12 KB to 8 KB (the single-CTA 128 x 256 tile is shared-memory-bandwidth bound:
// 96 B/clk of operand reads + 96 B/clk of TMA fills against 128 B/clk).  Accumulators: 128 lanes x BN columns in EACH
// CTA's TMEM, double buffered; each CTA's epilogue warps drain their own half.
// Barriers: full (leader only, tx bytes of BOTH CTAs), empty / tmem-full (commit multicast to both CTAs),
// tmem-empty (leader, 16 arrivals = 8 epilogue warps x 2 CTAs).
// ------------------------------------------------------------------------------------------------
// Tile rasterisation: tiles are walked in groups of GM row-tiles x all column-tiles (row fastest inside a group), so the
// ~74 tiles in flight at any time cover a GM x (74/GM) block: every A tile is shared by ~74/GM tiles and every B tile by GM
// tiles, instead of one B tile being requested by all SMs at once.
__device__ __forceinline__ void raster_tile(int t, int m_tiles, int n_tiles, int gm, int& mt, int& nt) {
  const int per_group = gm * n_tiles;
  const int g = t / per_group, r = t - g * per_group;
  const int m_in_group = min(gm, m_tiles - g * gm);
  mt = g * gm + r % m_in_group;
  nt = r / m_in_group;
}

template <int BN, bool SPLIT = false> struct Tc2Cfg {
  static constexpr int BM = 256, BMH = 128, BK = 64, UMMA_K = 16;
  static constexpr int A_BYTES = BMH * BK * 2;
  static constexpr int B_BYTES = (BN / 2) * BK * 2;
  static constexpr int HALVES = SPLIT ? 2 : 1;           // SPLIT: a stage holds [Ah | Wh | Al | Wl] of one K block
  static constexpr int STAGE_BYTES = HALVES * (A_BYTES + B_BYTES);
  static constexpr int STAGES = SPLIT ? ((BN == 256) ? 3 : 4) : ((BN == 256) ? 6 : 8);
  static constexpr int ACC_STAGES = 2;
  static constexpr int TMEM_COLS = ACC_STAGES * BN;
  static constexpr int BAR_BYTES = 256 + BN * 4;        // barriers + tmem slot, then the tile's bias (BN floats)
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + BAR_BYTES + 1024;
  static constexpr int EPI_WARPS = 8;                    // per CTA, warps 4..11: two per TMEM lane quarter, each takes every other 32-column chunk
  static constexpr int THREADS = 128 + EPI_WARPS * 32;   // warpgroup 0 = TMA producer, MMA issuer, TMEM allocator, one idle warp
  static_assert(BN == 128 || BN == 256, "BN");
};

template <int BN, typename TT, bool SPLIT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Tc2Cfg<BN, SPLIT>::THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const EpiParams ep, const int K) {
  using C = Tc2Cfg<BN, SPLIT>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tfull_bar = empty_bar + C::STAGES;
  uint64_t* tempty_bar = tfull_bar + C::ACC_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + C::ACC_STAGES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int num_kb = (K + C::BK - 1) / C::BK;
  const int m_tiles = (ep.M + C::BM - 1) / C::BM;
  const int n_tiles = (ep.N + BN - 1) / BN;
  const int ksplit = ep.ksplit > 1 ? ep.ksplit : 1;
  const int total_units = m_tiles * n_tiles * ksplit;           // unit = (tile, K slice); slices of a tile are consecutive units
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < C::STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < C::ACC_STAGES; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 2 * C::EPI_WARPS); }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc_cg2(tmem_slot, C::TMEM_COLS);
    tmem_relinquish_cg2();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                      // the peer's barriers exist before anything is signalled across the pair
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();

  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
  if (warp == 0) {
    // ===================== TMA producer (both CTAs; bytes are counted on the leader's full barrier) =====================
    if (lane == 0) {
      pdl_wait_prior_grid();
      int stage = 0; uint32_t phase = 0;
      for (int u = pair; u < total_units; u += n_pairs) {
        int mt, nt;
        raster_tile(u / ksplit, m_tiles, n_tiles, ep.raster_gm, mt, nt);
        const int ks = u % ksplit, kb_lo = ks * num_kb / ksplit, kb_hi = (ks + 1) * num_kb / ksplit;
        const int m0 = mt * C::BM + static_cast<int>(rank) * C::BMH;
        const int n0 = nt * BN + static_cast<int>(rank) * (BN / 2);
        for (int kb = kb_lo; kb < kb_hi; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * C::STAGE_BYTES;
          const uint32_t leader_full = mapa_u32(smem_u32(&full_bar[stage]), 0);
          if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * C::STAGE_BYTES);
          tma_load_2d_cg2(&tmA, leader_full, sa, kb * C::BK * C::HALVES, m0, kEvictNormal);
          tma_load_2d_cg2(&tmB, leader_full, sa + C::A_BYTES, kb * C::BK * C::HALVES, n0, kEvictNormal);
          if constexpr (SPLIT) {
            tma_load_2d_cg2(&tmA, leader_full, sa + C::A_BYTES + C::B_BYTES, kb * C::BK * 2 + C::BK, m0, kEvictNormal);
            tma_load_2d_cg2(&tmB, leader_full, sa + 2 * C::A_BYTES + C::B_BYTES, kb * C::BK * 2 + C::BK, n0, kEvictNormal);
          }
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (rank == 0 && lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16_f32(C::BM, BN);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int u = pair; u < total_units; u += n_pairs) {
        const int ks = u % ksplit, kb_lo = ks * num_kb / ksplit, kb_hi = (ks + 1) * num_kb / ksplit;
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);        // both CTAs' epilogues have drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = kb_lo; kb < kb_hi; ++kb) {
          mbar_wait(&full_bar[stage], phase);              // both CTAs' TMA bytes have landed
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * C::STAGE_BYTES);
          const uint64_t da = make_sw128_kmajor_desc(sa);
          const uint64_t db = make_sw128_kmajor_desc(sa + C::A_BYTES);
#pragma unroll
          for (int k = 0; k < C::BK / C::UMMA_K; ++k) umma_bf16_cg2(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb > kb_lo || k > 0) ? 1u : 0u);
          if constexpr (SPLIT) {                           // the lo products of the same K block: Ah.Wl + Al.Wh
            const uint64_t dal = make_sw128_kmajor_desc(sa + C::A_BYTES + C::B_BYTES), dbl = make_sw128_kmajor_desc(sa + 2 * C::A_BYTES + C::B_BYTES);
#pragma unroll
            for (int k = 0; k < C::BK / C::UMMA_K; ++k) {
              umma_bf16_cg2(d_tmem, da + 2 * k, dbl + 2 * k, idesc, 1u);
              umma_bf16_cg2(d_tmem, dal + 2 * k, db + 2 * k, idesc, 1u);
            }
          }
          umma_commit_cg2(&empty_bar[stage], 0b11);        // frees the slot in BOTH CTAs when these MMAs retire
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit_cg2(&tfull_bar[acc], 0b11);            // accumulator complete -> both epilogues
        if (++acc == C::ACC_STAGES) { acc = 0; acc_phase ^= 1; }
      }
    }
    __syncwarp();
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
    // ===================== epilogue warps: this CTA's 128 rows =====================
    // The epilogue of tile i runs under the MMAs of tile i+1, so it must stay shorter than one main loop (4.5 us at
    // K = 1024).  Everything it reads from global memory is therefore requested ahead of use: the tile's bias goes to smem
    // once, and the residual / gate / pos_embed operands of chunk c+1 are in flight while chunk c is computed (a first
    // version that loaded them inside the chunk loop took 12 us per tile and made the whole GEMM epilogue-bound).
    // Eight epilogue warps per CTA, two per TMEM lane quarter (warp % 4), each taking every other 32-column chunk of the tile: with
    // four - one per scheduler - the GELU and gate + residual epilogues took longer than the main loop and paced the GEMM.
    const int quarter = warp & 3;
    const int half = (warp - 4) >> 2;                       // 0: even chunks, 1: odd chunks
    constexpr int ET = C::EPI_WARPS * 32;
    const int et = threadIdx.x - 128;                       // 0..ET-1 among the epilogue threads
    float* bias_s = reinterpret_cast<float*>(tmem_slot + 4);   // BN floats behind the barriers
    pdl_wait_prior_grid();
    int acc = 0; uint32_t acc_phase = 0;
    for (int u = pair; u < total_units; u += n_pairs) {
      int mt, nt;
      raster_tile(u / ksplit, m_tiles, n_tiles, ep.raster_gm, mt, nt);
      const bool first_slice = (u % ksplit) == 0;            // the bias joins the sum exactly once
      const int m0 = mt * C::BM + static_cast<int>(rank) * C::BMH, n0 = nt * BN;
      const int m = m0 + quarter * 32 + lane;
      const bool row_ok = m < ep.M;
      const int mc = row_ok ? m : ep.M - 1;                 // clamped row: loads stay in bounds, stores are predicated
      named_bar_sync(1, ET);                                // previous tile's readers of bias_s are done
      for (int i = et; i < BN; i += ET) bias_s[i] = (ep.bias != nullptr && first_slice && n0 + i < ep.N) ? ep.bias[n0 + i] : 0.f;
      named_bar_sync(1, ET);
      constexpr int NCH = BN / 32;
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BN;
      if (ep.kind == EPI_GATE_RES) {
        float* xrow = reinterpret_cast<float*>(ep.out) + static_cast<size_t>(mc) * ep.ldo + n0;
        const TT* grow = reinterpret_cast<const TT*>(ep.gate) + static_cast<size_t>(ep.urow ? ep.urow[mc] : mc) * ep.ldg + ep.gate_off + n0;
        // Software pipeline over this warp's chunks: the residual and gate rows of chunk c+2 are requested as soon as those of chunk
        // c have been consumed (same registers), so they are in flight during the stores and the next TMEM load; the second warp of
        // the lane quarter covers the rest of the latency.  The gate row stays in the table's type while it is in flight.
        float4 xq[8];
        constexpr int GW = 32 * sizeof(TT) / 16;                            // 16-byte words per 32 gate values
        uint4 graw[GW];
        auto prefetch = [&](int c) {
          if (n0 + c * 32 < ep.N) {
            if (ksplit == 1) {
#pragma unroll
              for (int i = 0; i < 8; ++i) xq[i] = *reinterpret_cast<const float4*>(xrow + c * 32 + i * 4);
            }
#pragma unroll
            for (int i = 0; i < GW; ++i) graw[i] = reinterpret_cast<const uint4*>(grow + c * 32)[i];
          }
        };
        prefetch(half);
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
#pragma unroll 1
        for (int c = half; c < NCH; c += 2) {
          float v[32];
          tmem_ld32(t_addr + c * 32, v);
          tmem_ld_wait();
          const bool ok = row_ok && n0 + c * 32 < ep.N;
          float g[32];
          if constexpr (sizeof(TT) == 2) {
#pragma unroll
            for (int i = 0; i < GW; ++i) {
              const __nv_bfloat162* hp = reinterpret_cast<const __nv_bfloat162*>(&graw[i]);
#pragma unroll
              for (int k = 0; k < 4; ++k) { g[8 * i + 2 * k] = __low2float(hp[k]); g[8 * i + 2 * k + 1] = __high2float(hp[k]); }
            }
          } else {
#pragma unroll
            for (int i = 0; i < GW; ++i) { g[4 * i] = __uint_as_float(graw[i].x); g[4 * i + 1] = __uint_as_float(graw[i].y); g[4 * i + 2] = __uint_as_float(graw[i].z); g[4 * i + 3] = __uint_as_float(graw[i].w); }
          }
          if (ksplit > 1) {
            // K-sliced tile: x += gate * partial, summed in L2 by fp32 RED (the order of the slices is not fixed)
            if (c + 2 < NCH) prefetch(c + 2);
            if (ok) {
#pragma unroll
              for (int i = 0; i < 8; ++i)
                red_add_v4(xrow + c * 32 + i * 4, g[4 * i] * (v[4 * i] + bias_s[c * 32 + 4 * i]), g[4 * i + 1] * (v[4 * i + 1] + bias_s[c * 32 + 4 * i + 1]),
                           g[4 * i + 2] * (v[4 * i + 2] + bias_s[c * 32 + 4 * i + 2]), g[4 * i + 3] * (v[4 * i + 3] + bias_s[c * 32 + 4 * i + 3]));
            }
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) {                                   // x = x + gate * branch  (FMT.py:174-175), in place
              const float4 x = xq[i];
              v[4 * i] = fmaf(g[4 * i], v[4 * i] + bias_s[c * 32 + 4 * i], x.x);
              v[4 * i + 1] = fmaf(g[4 * i + 1], v[4 * i + 1] + bias_s[c * 32 + 4 * i + 1], x.y);
              v[4 * i + 2] = fmaf(g[4 * i + 2], v[4 * i + 2] + bias_s[c * 32 + 4 * i + 2], x.z);
              v[4 * i + 3] = fmaf(g[4 * i + 3], v[4 * i + 3] + bias_s[c * 32 + 4 * i + 3], x.w);
            }
            if (c + 2 < NCH) prefetch(c + 2);                               // the rows of this warp's next chunk, into the registers just consumed
            if (ok) store_row32(xrow + c * 32, v);
          }
        }
      } else {
        const float* prow = ep.kind == EPI_POS ? ep.pos + static_cast<size_t>(mc % ep.frames) * ep.N + n0 : nullptr;
        float4 pq[8];
        auto prefetch = [&](int c) {
          if (prow != nullptr && n0 + c * 32 < ep.N) {
#pragma unroll
            for (int i = 0; i < 8; ++i) pq[i] = *reinterpret_cast<const float4*>(prow + c * 32 + i * 4);
          }
        };
        prefetch(half);
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
#pragma unroll 1
        for (int c = half; c < NCH; c += 2) {
          float v[32];
          tmem_ld32(t_addr + c * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] += bias_s[c * 32 + i];
          if (ep.kind == EPI_GELU) {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = SPLIT ? gelu_tanh(v[i]) : gelu_tanh_approx(v[i]);   // tanh.approx: 2^-11, below the bf16 rounding of the output (not of a pair)
          } else if (ep.kind == EPI_POS) {
#pragma unroll
            for (int i = 0; i < 8; ++i) { v[4 * i] += pq[i].x; v[4 * i + 1] += pq[i].y; v[4 * i + 2] += pq[i].z; v[4 * i + 3] += pq[i].w; }
            if (c + 2 < NCH) prefetch(c + 2);
          }
          if (row_ok && n0 + c * 32 < ep.N) {
            if (ep.out_f32) store_row32(reinterpret_cast<float*>(ep.out) + static_cast<size_t>(m) * ep.ldo + n0 + c * 32, v);
            else if constexpr (SPLIT) VecIO<bf16x3_t, 32>::store(reinterpret_cast<bf16x3_t*>(ep.out) + static_cast<size_t>(m) * ep.ldo + n0 + c * 32, v);
            else store_row32(reinterpret_cast<__nv_bfloat16*>(ep.out) + static_cast<size_t>(m) * ep.ldo + n0 + c * 32, v);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty_bar[acc]), 0));
      if (++acc == C::ACC_STAGES) { acc = 0; acc_phase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                      // nobody leaves while the peer may still read this CTA's smem or signal its barriers
  if (warp == 2) tmem_dealloc_cg2(tmem_base, C::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------
// fp32 SIMT GEMM (validation mode).  64x64 tile, K step 16, 256 threads x (4x4) outputs.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gemm_simt_kernel(const float* __restrict__ A, int lda, const float* __restrict__ W, int ldw,
                                                        const EpiParams ep, const int K) {
  __shared__ float sA[16][64 + 4];
  __shared__ float sW[16][64 + 4];
  pdl_launch_dependents();
  pdl_wait_prior_grid();
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
    // each thread loads one float4 of A and one of W: row = tid/4 (0..63), k-quad = tid%4
    const int r = threadIdx.x >> 2, kq = (threadIdx.x & 3) * 4;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), w = a;
    if (m0 + r < ep.M) a = *reinterpret_cast<const float4*>(A + static_cast<size_t>(m0 + r) * lda + k0 + kq);
    if (n0 + r < ep.N) w = *reinterpret_cast<const float4*>(W + static_cast<size_t>(n0 + r) * ldw + k0 + kq);
    sA[kq][r] = a.x; sA[kq + 1][r] = a.y; sA[kq + 2][r] = a.z; sA[kq + 3][r] = a.w;
    sW[kq][r] = w.x; sW[kq + 1][r] = w.y; sW[kq + 2][r] = w.z; sW[kq + 3][r] = w.w;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float av[4], wv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { av[i] = sA[k][ty * 4 + i]; wv[i] = sW[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i, n = n0 + tx * 4;
    if (m < ep.M && n < ep.N) epi_apply<float, float, 4>(ep, m, n, acc[i]);
  }
}

}  // namespace fmt
