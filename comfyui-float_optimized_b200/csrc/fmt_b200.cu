// libfmt_b200.so - host side of the C ABI declared in include/fmt_b200.h.
//
// Owns: the packed weights (bf16 for the tcgen05 path, fp32 for the validation mode, bf16x3 pairs once a plan selects that
// mode), the workspace, the per-plan CUDA graph of one sampling window, and the window loop of _perform_ode_sampling_loop
// (nodes_adv.py:545-694), which runs entirely on the device: windows are chained through prev_x / prev_wa / prev_we without host syncs.
#include "../../include/fmt_b200.h"
#include "kernels.cuh"
#include "window.cuh"
#include "flow.cuh"
#include "stages.cuh"

#include <algorithm>
#include <functional>
#include <map>
#include <queue>
#include <tuple>
#include <cstdlib>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

using namespace fmt;
typedef __nv_bfloat16 bf16;

// ------------------------------------------------------------------------------------------------ errors
static thread_local char g_err[1024] = "";
static int set_err(int code, const char* fmtstr, ...) {
  va_list ap;
  va_start(ap, fmtstr);
  vsnprintf(g_err, sizeof(g_err), fmtstr, ap);
  va_end(ap);
  return code;
}
#define CUDA_OK(expr)                                                                                         \
  do {                                                                                                        \
    cudaError_t _e = (expr);                                                                                  \
    if (_e != cudaSuccess) return set_err(-2, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)
#define FMT_OK(expr)          \
  do {                        \
    int _r = (expr);          \
    if (_r != 0) return _r;   \
  } while (0)
#define REQUIRE(cond, ...)                          \
  do {                                              \
    if (!(cond)) return set_err(-1, __VA_ARGS__);   \
  } while (0)

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// ------------------------------------------------------------------------------------------------ handle
struct Linear {
  bf16* w16 = nullptr;    // (N, K) bf16, K possibly padded
  float* w32 = nullptr;   // (N, K) fp32 (validation mode)
  bf16* w3 = nullptr;     // (N, 2K) bf16x3 pairs (gemm.cuh), packed from w32 the first time a plan or projection selects FMT_MODE_BF16X3
  float* b = nullptr;     // (N)
  int N = 0, K = 0;
};

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
};

struct FmtHandle {
  int device = 0;
  int num_sms = 148;
  FmtDims d{};
  int N = 0, Kc = 0, NT = 0;
  PFN_encodeTiled encode = nullptr;

  Linear x_emb, c_emb, ada, dec;
  std::vector<Linear> qkv, proj, fc1, fc2;
  float *t0_w = nullptr, *t0_b = nullptr, *t2_w = nullptr, *t2_b = nullptr, *pos = nullptr;
  std::vector<void*> owned;

  // plan
  bool configured = false;
  FmtPlan plan{};
  std::vector<float> t_eval, dt, rk_a, rk_b;
  ModelShape shape{};
  int R = 0, U = 0, n_eval = 0, table_chunk = 0;
  size_t tsize = 2;   // sizeof(activation type)

  // workspace
  DevBuf cond, cemb, temb, tfreq, th, silu, table, xstate, ystage, kbuf, prevx, ax, X, A1, QKV, A2, Hm, V, ddt, dteval, wargs;
  DevBuf urow_buf, uidx_buf;                     // condition-row deduplication: table row of every token row / token row each table row stands for
  bool dedup = false;                            // U < R: the AdaLN tables hold one row per DISTINCT condition row (FMT_DEDUP=0 switches it off)
  int use_dedup = 1;
  DevBuf st_rs, st_wa, st_we, st_noise, st_rd;   // staging for host-located clips
  DevBuf ev_wa, ev_we;                           // fmt_velocity: [prev_wa | wa] and [prev_we | we] of every clip, (B, P + L, .)
  // the slot records of every window of a sampling call ([window][slot]), uploaded with one copy from a pinned staging
  // buffer; slot_ev marks the end of that copy, so the next call waits for it before it refills the staging buffer.  A window's
  // records are slot_stride bytes: one SlotArgs per slot of the graph it replays, followed by as many SlotOde in calls of the per-slot
// window graph.
  DevBuf slot_buf, slot_zero;                    // slot_zero: the inputs of an idle slot
  unsigned char* slot_host = nullptr;
  size_t slot_host_bytes = 0, slot_stride = 0;
  int slot_recs = 0;                             // records per window of the staged call
  cudaEvent_t slot_ev = nullptr;
  // per-slot ODE schedules (fmt_sample_clips_ode, fmt_sample_windows_ode): a second window graph of the plan, captured on first use.
  // It shares the plan's workspace and AdaLN table buffer; its condition rows never span two slots (sU rows, sU - U more than the
  // plan's in 4-branch plans), its kbuf holds FMT_MAX_STAGES stages.
  std::map<std::vector<float>, DevBuf> ode_cache;   // t-embeddings and step sizes of every schedule seen, keyed by its contents
  DevBuf s_cond, s_cemb, s_urow, s_uidx, s_kbuf;
  int sU = 0, s_chunk = 0;
  bool s_dedup = false;
  cudaGraphExec_t ode_exec = nullptr;
  int ode_nodes = 0;
  long long ode_launches = 0;
  bool last_ode = false;                         // the last sampling call ran the per-slot graph
  bool use_splitk = false;                       // 2-way K slicing of gate+residual GEMMs with a ragged last wave (FMT_SPLITK=1; measured 3 % slower at 32 clips)
  int raster_gm = 8;                             // FMT_RASTER_GM
  bool use_pair = true;                          // CTA-pair (cta_group::2) GEMM for M >= 512 (FMT_PAIR=0 disables)
  bool use_pdl = true;                           // programmatic dependent launch between graph nodes (FMT_PDL=0 disables)
  size_t ws_bytes = 0;

  // persistent window kernel (window.cuh): used when the plan has <= 256 token rows in bf16 mode
  int use_window = 3;                            // FMT_WINDOW: 0 = one kernel per op, 1 = barrier-stepped split-K window kernel, 2 = grouped one, 3 = dataflow kernel (flow.cuh)
  bool window_active = false;
  // dataflow window kernel (flow.cuh)
  bool flow_active = false;
  int flow_ch = 64;                              // rows per chunk (FMT_FLOW_CH = 32 | 64)
  int flow_max_rows = 256;                       // plans with more token rows run one kernel per op (FMT_FLOW_MAX_ROWS)
  int flow_fixed = 14;                           // FMT_FLOW_FIXED: split-K partial sums are rounded to multiples of 2^-k before they meet in L2 (exact, order-independent sums below 2^(24-k): bitwise reproducible runs); 0 = off
  int flow_poll = 1;                             // FMT_FLOW_POLL: 0 = acquire polls, 1 = relaxed polls + one acquire load
  long long flow_spin_limit = 20000000000ll;     // SM clocks (~10 s) a wait may spin before the kernel traps (FMT_FLOW_SPIN_MS): long enough to survive a time-sliced GPU, short enough to end a protocol bug
  FlowParams flow_params{};
  DevBuf flow_gemms, flow_tmaps, flow_acc, flow_act, flow_flags, flow_trace;
  bool win_grouped = false;                      // the active plan runs fmt_window_kernel<NV, true>
  int win_spg = 1;                               // sequences per group (FMT_WIN_SPG), rows per group = spg * N <= 128
  int win_fuse_gelu = 1;                         // FMT_WIN_FUSE_GELU=0 keeps the separate GELU stage in the grouped schedule
  int win_nf[4] = {0, 0, 0, 0};                  // feature-slice overrides for qkv / proj / fc1 / fc2 (FMT_WIN_NF; 0 = auto)
  int win_pk[4] = {0, 0, 0, 0};                  // K-split overrides for qkv / proj / fc1 / fc2 (FMT_WIN_PK="q,p,1,2"; 0 = auto)
  DevBuf win_params, win_tmaps, win_acc, win_bar, win_trace, win_act;   // win_act: pre-tiled A1 | A2 | Hm operands
  int win_trace_stride = 0;
  int* win_err_host = nullptr;                   // mapped pinned int: which bounded spin tripped (0 = none)
  int* win_err_dev = nullptr;

  cudaGraphExec_t graph_exec = nullptr;
  int graph_nodes = 0;
  long long launches = 0;
  bool capturing = false;
  long long capture_launches = 0;
  bool ksliced = false;                          // a graph captured since the flag was cleared cuts a GEMM into K slices

  // occupancy buckets of a plan whose window graph runs one kernel per op (fmt_sample_window_set): a step with k ready streams
  // replays graphs captured for fmt_occupancy_slots(batch, k) slots.  Bucket i (of 2^i slots, below batch) gets its condition-row
  // map in fmt_configure and its graphs on first use; the plan's own graphs serve the bucket of batch slots.
  struct Bucket {
    int B = 0, U = 0;                            // slots, distinct condition rows of the plan's graph for them
    size_t map_off = 0;                          // its urow (R ints) | uidx (U ints) in bucket_maps
    cudaGraphExec_t exec = nullptr;
    long long launches = 0;
    int sU = 0;                                  // the per-slot window graph's: condition rows, map (built on first use), graph
    DevBuf s_map;
    cudaGraphExec_t ode_exec = nullptr;
    long long ode_launches = 0;
  };
  std::vector<Bucket> buckets;
  DevBuf bucket_maps;
  bool plan_ksliced = false;                     // the plan's window graph cuts a GEMM into K slices: its buckets may too
  int last_slots = 0;                            // slots of the last window graph replayed
};

static int dev_alloc(FmtHandle* h, DevBuf& b, size_t bytes) {
  if (b.bytes >= bytes && b.p) return 0;
  if (b.p) {
    CUDA_OK(cudaFree(b.p));
    h->ws_bytes -= b.bytes;
    b.p = nullptr;
    b.bytes = 0;
  }
  bytes = (bytes + 255) & ~static_cast<size_t>(255);
  CUDA_OK(cudaMalloc(&b.p, bytes));
  b.bytes = bytes;
  h->ws_bytes += bytes;
  return 0;
}

static inline void count_launch(FmtHandle* h) {
  if (h->capturing) h->capture_launches++;
  else h->launches++;
}
#define LAUNCH_CHECK() CUDA_OK(cudaGetLastError())

// All kernels of the step go through here: optional thread-block cluster + programmatic dependent launch, so that in the
// captured graph the prologue (barrier init, TMEM alloc, weight prefetch) of node i+1 overlaps the tail of node i.
template <typename... KArgs, typename... Args>
static int launch(FmtHandle* h, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attrs[2];
  int na = 0;
  if (cluster > 1) {
    attrs[na].id = cudaLaunchAttributeClusterDimension;
    attrs[na].val.clusterDim.x = cluster; attrs[na].val.clusterDim.y = 1; attrs[na].val.clusterDim.z = 1;
    ++na;
  }
  if (h->use_pdl) {
    attrs[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attrs[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attrs; cfg.numAttrs = na;
  CUDA_OK(cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...));
  count_launch(h);
  return 0;
}

// ------------------------------------------------------------------------------------------------ GEMM launch
static int make_tmap(FmtHandle* h, CUtensorMap* m, const void* ptr, int rows, int cols, int ld_elems, int box_rows) {
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld_elems) * 2};
  cuuint32_t box[2] = {64, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = h->encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_err(-3, "cuTensorMapEncodeTiled failed (%d) rows=%d cols=%d ld=%d box=%d ptr=%p", (int)r, rows, cols, ld_elems, box_rows, ptr);
  return 0;
}

static int make_tmap_ex(FmtHandle* h, CUtensorMap* m, const void* ptr, CUtensorMapDataType dt, int elem_bytes, int rows, int cols, int ld_elems,
                        int box_cols, int box_rows, CUtensorMapSwizzle sw) {
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld_elems) * elem_bytes};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = h->encode(m, dt, 2, const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_err(-3, "cuTensorMapEncodeTiled failed (%d) rows=%d cols=%d ld=%d box=%dx%d ptr=%p", (int)r, rows, cols, ld_elems, box_cols, box_rows, ptr);
  return 0;
}

// SPLIT (FMT_MODE_BF16X3): A and W are pair matrices (gemm.cuh), lda / ldw / K count logical columns; the tensor maps cover the
// 2K bf16 columns of their rows.  Gate tables are fp32 in that mode.
template <int BN, bool SPLIT>
static int launch_tc(FmtHandle* h, const bf16* A, int lda, const bf16* W, int ldw, const EpiParams& ep, int K, cudaStream_t st) {
  using C = TcCfg<BN, SPLIT>;
  const auto kern = gemm_tc_kernel<BN, typename std::conditional<SPLIT, float, bf16>::type, SPLIT>;
  static bool attr_set[64] = {};
  if (!attr_set[h->device & 63]) {   // per device: the attribute lives in the device's module image
    CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    attr_set[h->device & 63] = true;
  }
  CUtensorMap ta, tb;
  FMT_OK(make_tmap(h, &ta, A, ep.M, K * C::HALVES, lda * C::HALVES, C::BM));
  FMT_OK(make_tmap(h, &tb, W, ep.N, K * C::HALVES, ldw * C::HALVES, BN));
  const int tiles = ((ep.M + C::BM - 1) / C::BM) * ((ep.N + BN - 1) / BN);
  const int grid = tiles < h->num_sms ? tiles : h->num_sms;
  return launch(h, kern, dim3(grid), dim3(C::THREADS), C::SMEM_BYTES, st, 1, ta, tb, ep, K);
}

template <int BN, bool SPLIT>
static int launch_tc2(FmtHandle* h, const bf16* A, int lda, const bf16* W, int ldw, const EpiParams& ep, int K, cudaStream_t st, int ksplit = 1) {
  using C = Tc2Cfg<BN, SPLIT>;
  // every K slice must hold a K block: an empty slice issues no MMA, and its epilogue would add a stale accumulator into x
  REQUIRE(ksplit == 1 || (ksplit > 1 && ep.kind == EPI_GATE_RES && K >= 64 * ksplit), "gemm: %d K slices need x += gate * (.) and K >= %d (K=%d)",
          ksplit, 64 * ksplit, K);
  const auto kern = gemm_tc2_kernel<BN, typename std::conditional<SPLIT, float, bf16>::type, SPLIT>;
  static bool attr_set[64] = {};
  if (!attr_set[h->device & 63]) {
    CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    attr_set[h->device & 63] = true;
  }
  CUtensorMap ta, tb;
  FMT_OK(make_tmap(h, &ta, A, ep.M, K * C::HALVES, lda * C::HALVES, C::BMH));
  FMT_OK(make_tmap(h, &tb, W, ep.N, K * C::HALVES, ldw * C::HALVES, BN / 2));
  const int tiles = ((ep.M + C::BM - 1) / C::BM) * ((ep.N + BN - 1) / BN) * ksplit;
  const int max_pairs = h->num_sms / 2;
  const int pairs = tiles < max_pairs ? tiles : max_pairs;
  EpiParams ep2 = ep;
  ep2.raster_gm = h->raster_gm;
  ep2.ksplit = ksplit;
  // the kernel carries __cluster_dims__(2,1,1); launch() only adds the PDL attribute
  return launch(h, kern, dim3(2 * pairs), dim3(C::THREADS), C::SMEM_BYTES, st, 1, ta, tb, ep2, K);
}

static int pick_bn(const FmtHandle* h, int M, int N) {
  const int mt = (M + 127) / 128;
  if (N % 256 == 0 && mt * (N / 256) >= 2 * h->num_sms) return 256;
  if (N % 128 == 0 && mt * (N / 128) >= h->num_sms) return 128;
  return 64;
}

// SPLIT: the bf16x3 GEMM on pair operands (FMT_MODE_BF16X3): K % 64 == 0, never K-sliced by the sampler (its results stay bitwise
// reproducible).  force_ksplit: K slices of a forced CTA-pair kernel (unit tests); the sampler picks them itself where ksplit allows it
// (a window graph's GraphShape::ksplit).  Every other choice of kernel and tile gives the same bits (tests/test_gpu_gemm_variants.py).
template <bool SPLIT = false>
static int gemm_bf16(FmtHandle* h, const bf16* A, int lda, const bf16* W, int ldw, const EpiParams& ep, int K, cudaStream_t st, int force_bn = 0,
                     int force_ksplit = 1, bool ksplit = false) {
  REQUIRE(ep.N % 32 == 0 && K % 8 == 0 && lda % 8 == 0 && ldw % 8 == 0, "gemm_bf16: N %% 32, K/lda/ldw %% 8 required (N=%d K=%d)", ep.N, K);
  REQUIRE(!SPLIT || (K % 64 == 0 && lda % 64 == 0 && ldw % 64 == 0), "gemm_bf16x3: K, lda, ldw %% 64 required (K=%d)", K);
  REQUIRE(force_ksplit == 1 || force_bn == 512 || force_bn == 1024, "gemm_bf16: K slices need the CTA-pair kernel (block_n 512 or 1024)");
  // CTA-pair kernel (force_bn 512 / 1024 = pair tiles 256x256 / 256x128): the default once there are enough 256-row tiles
  if (force_bn == 512) return launch_tc2<256, SPLIT>(h, A, lda, W, ldw, ep, K, st, force_ksplit);
  if (force_bn == 1024) return launch_tc2<128, SPLIT>(h, A, lda, W, ldw, ep, K, st, force_ksplit);
  if (force_bn == 0 && h->use_pair && ep.M >= 512 && ep.N % 256 == 0 && K % 64 == 0) {
    // Wave model calibrated on B200 (tools/gemm_bench.py): time ~ waves x per-wave cost.  A pair tile (256x256 on two SMs)
    // and a single-CTA 128x256 tile cost the same per wave at 32 clips, but at >= 128 clips the pair kernel is 20 % cheaper
    // (half the L2 -> SM operand traffic); a 128x128 tile costs 0.56 of a wave and wins when the wider tiles leave the last
    // wave mostly empty (N = 1024 at 32 clips: 92 pair tiles on 74 pairs).
    const int sms = h->num_sms, pairs = sms / 2, mt128 = (ep.M + 127) / 128, mt256 = (ep.M + 255) / 256;
    const auto waves = [](int tiles, int units) { return static_cast<double>((tiles + units - 1) / units); };
    const double c_pair = waves(mt256 * (ep.N / 256), pairs);
    const double c_256 = waves(mt128 * (ep.N / 256), sms) * (ep.M >= 16384 ? 1.2 : 1.02);
    const double c_128 = waves(mt128 * (ep.N / 128), sms) * 0.56;
    // bf16x3: the same model (its operand bytes and MMAs both grow ~2-3x on every tile shape); a single-CTA 128 x 256 tile would
    // keep only 2 of its 96 KB stages, so the pair tile or 128 x 128 it is
    if (SPLIT) return c_pair <= c_128 ? launch_tc2<256, true>(h, A, lda, W, ldw, ep, K, st) : launch_tc<128, true>(h, A, lda, W, ldw, ep, K, st);
    if (ep.kind == EPI_GATE_RES && ksplit && K >= 1024 && c_pair >= 2.0) {   // single-wave problems stay bitwise deterministic
      // x += gate * (.) is additive, so a tile may be cut into 2 K slices whose partial sums meet in x (fp32 RED):
      // N = 1024 at 32 clips = 92 pair tiles on 74 pairs (2 waves) -> 184 half-K units (2.5 half-waves)
      const double c_split = 0.5 * waves(2 * mt256 * (ep.N / 256), pairs) + 0.08;
      if (c_split < c_pair && c_split < c_256 && c_split < c_128) {
        if (h->capturing) h->ksliced = true;
        return launch_tc2<256, false>(h, A, lda, W, ldw, ep, K, st, 2);
      }
    }
    if (c_pair <= c_256 && c_pair <= c_128) return launch_tc2<256, false>(h, A, lda, W, ldw, ep, K, st);
    return c_128 < c_256 ? launch_tc<128, false>(h, A, lda, W, ldw, ep, K, st) : launch_tc<256, false>(h, A, lda, W, ldw, ep, K, st);
  }
  int bn = force_bn > 0 ? force_bn : pick_bn(h, ep.M, ep.N);
  if (SPLIT && force_bn == 0 && bn == 256) bn = 128;      // 2 stages of 96 KB: explicit block_n only
  switch (bn) {
    case 256: return launch_tc<256, SPLIT>(h, A, lda, W, ldw, ep, K, st);
    case 128: return launch_tc<128, SPLIT>(h, A, lda, W, ldw, ep, K, st);
    case 64: return launch_tc<64, SPLIT>(h, A, lda, W, ldw, ep, K, st);
  }
  return set_err(-1, "gemm_bf16: block_n must be 64, 128 or 256 (got %d)", bn);
}

static int gemm_f32(FmtHandle* h, const float* A, int lda, const float* W, int ldw, const EpiParams& ep, int K, cudaStream_t st) {
  REQUIRE(ep.N % 4 == 0 && K % 16 == 0 && lda % 4 == 0 && ldw % 4 == 0, "gemm_f32: N %% 4, K %% 16 required (N=%d K=%d)", ep.N, K);
  dim3 grid((ep.N + 63) / 64, (ep.M + 63) / 64);
  return launch(h, gemm_simt_kernel, grid, dim3(256), 0, st, 1, A, lda, W, ldw, ep, K);
}

// T = GEMM operand (activation) type of a mode; Tab = type of its AdaLN tables and of QKV
template <typename T> struct ModeOps;
template <> struct ModeOps<bf16> {
  using Tab = bf16;
  static int gemm(FmtHandle* h, const void* A, int lda, const Linear& L, const EpiParams& ep, bool ksplit, cudaStream_t st) {
    return gemm_bf16(h, static_cast<const bf16*>(A), lda, L.w16, L.K, ep, L.K, st, 0, 1, ksplit);
  }
};
template <> struct ModeOps<float> {
  using Tab = float;
  static int gemm(FmtHandle* h, const void* A, int lda, const Linear& L, const EpiParams& ep, bool, cudaStream_t st) {
    return gemm_f32(h, static_cast<const float*>(A), lda, L.w32, L.K, ep, L.K, st);
  }
};
template <> struct ModeOps<bf16x3_t> {
  using Tab = float;                                   // only GEMM operands are pairs: tables and QKV stay fp32, as in the fp32 mode
  static int gemm(FmtHandle* h, const void* A, int lda, const Linear& L, const EpiParams& ep, bool, cudaStream_t st) {
    return gemm_bf16<true>(h, static_cast<const bf16*>(A), lda, L.w3, L.K, ep, L.K, st);
  }
};

static EpiParams epi(int kind, int M, int N, const float* bias, void* out, int ldo, int out_f32) {
  EpiParams p{};
  p.kind = kind; p.M = M; p.N = N; p.bias = bias; p.out = out; p.ldo = ldo; p.out_f32 = out_f32;
  return p;
}

// ------------------------------------------------------------------------------------------------ the FMT step
// The distinct condition rows a window graph works on: the plan's (fmt_configure), or the per-slot graph's, which never shares a row
// between two slots.  urow / uidx: table row of every token row / token row of every table row (nullptr: the identity).
struct CondRows {
  int U;
  const int* urow;
  const int* uidx;
  void* cond;
  void* cemb;
  int chunk;                                     // evaluations whose tables the table buffer holds at once
  bool per_slot;                                 // t-embeddings of each slot's own schedule (silu_cond_sched_kernel)
};

static CondRows plan_rows(const FmtHandle* h) {
  return CondRows{h->U, h->dedup ? static_cast<const int*>(h->urow_buf.p) : nullptr, h->dedup ? static_cast<const int*>(h->uidx_buf.p) : nullptr,
                  h->cond.p, h->cemb.p, h->table_chunk, false};
}

static CondRows ode_rows(const FmtHandle* h) {
  return CondRows{h->sU, h->s_dedup ? static_cast<const int*>(h->s_urow.p) : nullptr, h->s_dedup ? static_cast<const int*>(h->s_uidx.p) : nullptr,
                  h->s_cond.p, h->s_cemb.p, h->s_chunk, true};
}

// Band attention of n_seq sequences of N rows.  variant 0 picks the kernel, 1 forces the warp-per-row kernel, 2 the tile kernel.
enum { ATTN_AUTO = 0, ATTN_WARP = 1, ATTN_TILE = 2 };

// What one captured window graph works on.  The plan's graphs run all plan.batch slots; an occupancy bucket's graphs
// (fmt_sample_window_set) run the first B of them, on a prefix of every workspace buffer.  A bucket keeps whatever changes the bits of
// a slot's rows: the band-attention kernel (the tile and the warp-per-row kernel reduce in different orders, and the plan's choice
// depends on its sequence count) and K slicing (its partial sums meet in x in any order).  It picks its own GEMM tiles: every tile
// shape and the CTA-pair kernel compute each output element the same way.
struct GraphShape {
  ModelShape s;                                  // s.B: the graph's slots
  int R;                                         // token rows, s.nb * s.B * s.N
  CondRows rows;                                 // condition rows of those slots (the plan's table_chunk, so the same node count)
  int attn;                                      // ATTN_WARP or ATTN_TILE: the plan's
  bool ksplit;                                   // gate + residual GEMMs may be cut into K slices
};

// the band-attention kernel ATTN_AUTO picks for n_seq sequences of the model in this activation type
static int attn_variant(const FmtHandle* h, bool bf16_act, int n_seq) {
  const int hd = h->d.dim_h / h->d.num_heads;
  const bool tile_ok = bf16_act && static_cast<size_t>(2) * h->N * hd * sizeof(bf16) <= 48 * 1024 && (hd == 64 || hd == 128);
  return tile_ok && n_seq * h->d.num_heads >= 2 * h->num_sms ? ATTN_TILE : ATTN_WARP;
}

// the plan's window graph (ode: its per-slot window graph)
static GraphShape plan_graph(const FmtHandle* h, bool ode = false) {
  return GraphShape{h->shape, h->R, ode ? ode_rows(h) : plan_rows(h), attn_variant(h, h->plan.mode == FMT_MODE_BF16, h->shape.nb * h->shape.B),
                    h->use_splitk};
}

template <typename T>
static int enqueue_prepare(FmtHandle* h, const GraphShape& g, cudaStream_t st) {
  const ModelShape& s = g.s;
  const CondRows& r = g.rows;
  const WindowArgs* wa = static_cast<const WindowArgs*>(h->wargs.p);
  FMT_OK(launch(h, cond_gather_kernel<T>, dim3(r.U), dim3(128), 0, st, 1, wa, s, r.uidx, static_cast<T*>(r.cond)));
  EpiParams ep = epi(EPI_STORE, r.U, s.H, h->c_emb.b, r.cemb, s.H, 1);
  FMT_OK(ModeOps<T>::gemm(h, r.cond, s.Kc, h->c_emb, ep, g.ksplit, st));
  return 0;
}

// AdaLN tables for evaluations [e0, e0+n): table[(e-e0)*U + u, :] = Linear_ada(SiLU(c_emb[u] + t_emb[e]))
template <typename T>
static int enqueue_tables(FmtHandle* h, const GraphShape& g, int e0, int n, cudaStream_t st) {
  const ModelShape& s = g.s;
  const CondRows& r = g.rows;
  const size_t total = static_cast<size_t>(n) * r.U * s.H;
  const dim3 grid(static_cast<unsigned>((total / 4 + 255) / 256));
  if (r.per_slot)
    FMT_OK(launch(h, silu_cond_sched_kernel<T>, grid, dim3(256), 0, st, 1, static_cast<const WindowArgs*>(h->wargs.p), s,
                  static_cast<const float*>(r.cemb), r.uidx, e0, r.U, static_cast<T*>(h->silu.p), total));
  else
    FMT_OK(launch(h, silu_cond_kernel<T>, grid, dim3(256), 0, st, 1, static_cast<const float*>(r.cemb), static_cast<const float*>(h->temb.p), e0,
                  r.U, s.H, static_cast<T*>(h->silu.p), total));
  EpiParams ep = epi(EPI_STORE, n * r.U, h->NT, h->ada.b, h->table.p, h->NT, sizeof(typename ModeOps<T>::Tab) == 4);
  FMT_OK(ModeOps<T>::gemm(h, h->silu.p, s.H, h->ada, ep, g.ksplit, st));
  return 0;
}

// LayerNorm + modulate of `rows` rows of X into out (the GEMM operand of the next Linear); table rows are urow[r] (NULL = r) * ldt
template <typename T>
static int lnmod(FmtHandle* h, const float* X, int rows, int H, const typename ModeOps<T>::Tab* table, const int* urow, long long ldt,
                 long long shift_off, long long scale_off, T* out, cudaStream_t st) {
  using TT = typename ModeOps<T>::Tab;
  const int warps = 4;
  const dim3 grid((rows + warps - 1) / warps), block(warps * 32);
  switch (H % 128 == 0 ? H / 128 : 0) {
    case 1: return launch(h, lnmod_kernel<T, TT, 1>, grid, block, 0, st, 1, X, rows, H, table, urow, ldt, shift_off, scale_off, out);
    case 2: return launch(h, lnmod_kernel<T, TT, 2>, grid, block, 0, st, 1, X, rows, H, table, urow, ldt, shift_off, scale_off, out);
    case 4: return launch(h, lnmod_kernel<T, TT, 4>, grid, block, 0, st, 1, X, rows, H, table, urow, ldt, shift_off, scale_off, out);
    case 8: return launch(h, lnmod_kernel<T, TT, 8>, grid, block, 0, st, 1, X, rows, H, table, urow, ldt, shift_off, scale_off, out);
  }
  return set_err(-1, "dim_h %d unsupported by the LayerNorm kernel (128, 256, 512, 1024)", H);
}

template <typename T>
static int launch_lnmod(FmtHandle* h, const GraphShape& g, const typename ModeOps<T>::Tab* table_e, long long shift_off, long long scale_off,
                        cudaStream_t st) {
  return lnmod<T>(h, static_cast<const float*>(h->X.p), g.R, g.s.H, table_e, g.rows.urow, h->NT, shift_off, scale_off, static_cast<T*>(h->A1.p), st);
}

template <typename T>
static int band_attention(FmtHandle* h, const typename ModeOps<T>::Tab* qkv, int n_seq, int N, int heads, int hd, int win, T* out, int variant,
                          cudaStream_t st) {
  using Q = typename ModeOps<T>::Tab;
  const float scale = 1.0f / sqrtf(static_cast<float>(hd));
  // many sequences: one CTA per (sequence, head) with K / V staged in shared memory (every qkv byte read once)
  const size_t tile_smem = static_cast<size_t>(2) * N * hd * sizeof(bf16);   // K, V of one (sequence, head)
  const bool tile_ok = sizeof(T) == 2 && tile_smem <= 48 * 1024 && (hd == 64 || hd == 128);
  if (variant == ATTN_AUTO) variant = tile_ok && n_seq * heads >= 2 * h->num_sms ? ATTN_TILE : ATTN_WARP;
  if (variant == ATTN_TILE) {
    REQUIRE(tile_ok, "band attention: the tile kernel needs bf16, head_dim 64 or 128 and K / V within 48 KB (N=%d hd=%d)", N, hd);
    if constexpr (sizeof(T) == 2) {
      const bf16* q16 = reinterpret_cast<const bf16*>(qkv);
      bf16* o16 = reinterpret_cast<bf16*>(out);
      const dim3 tg(n_seq * heads), tb(ATTN_TILE_THREADS);
      if (hd == 64) return launch(h, band_attention_tile_kernel<64>, tg, tb, tile_smem, st, 1, q16, N, heads, win, scale, o16);
      return launch(h, band_attention_tile_kernel<128>, tg, tb, tile_smem, st, 1, q16, N, heads, win, scale, o16);
    }
  }
  REQUIRE(variant == ATTN_WARP, "band attention: unknown variant %d", variant);
  const int total_warps = n_seq * heads * N, warps = 4;
  const dim3 grid((total_warps + warps - 1) / warps), block(warps * 32);
  switch (hd) {
    case 32: return launch(h, band_attention_kernel<Q, 1, T>, grid, block, 0, st, 1, qkv, n_seq, N, heads, win, scale, out);
    case 64: return launch(h, band_attention_kernel<Q, 2, T>, grid, block, 0, st, 1, qkv, n_seq, N, heads, win, scale, out);
    case 128: return launch(h, band_attention_kernel<Q, 4, T>, grid, block, 0, st, 1, qkv, n_seq, N, heads, win, scale, out);
  }
  return set_err(-1, "head_dim %d unsupported (32, 64, 128)", hd);
}

template <typename T>
static int launch_attn(FmtHandle* h, const GraphShape& g, cudaStream_t st) {
  const ModelShape& s = g.s;
  const int heads = h->d.num_heads;
  return band_attention<T>(h, static_cast<const typename ModeOps<T>::Tab*>(h->QKV.p), s.nb * s.B, s.N, heads, s.H / heads, h->d.attention_window,
                           static_cast<T*>(h->A2.p), g.attn, st);
}

// One model evaluation: V[R, W] = FMT.forward over the nb-way batched CFG branches (FMT.py:277-340).  The x-embedder
// operand `ax` has already been written by the producer of the ODE state (init_window / cfg_combine / rk_combine).
template <typename T>
static int enqueue_forward(FmtHandle* h, const GraphShape& g, int table_slot, cudaStream_t st) {
  const ModelShape& s = g.s;
  const CondRows& r = g.rows;
  const FmtDims& d = h->d;
  const int R = g.R, H = s.H;
  const bool ks = g.ksplit;
  using TT = typename ModeOps<T>::Tab;
  const TT* table_e = static_cast<const TT*>(h->table.p) + static_cast<size_t>(table_slot) * r.U * h->NT;
  const int qkv_f32 = sizeof(TT) == 4;
  {
    EpiParams ep = epi(EPI_POS, R, H, h->x_emb.b, h->X.p, H, 1);
    ep.pos = h->pos; ep.frames = s.N;
    FMT_OK(ModeOps<T>::gemm(h, h->ax.p, s.W, h->x_emb, ep, ks, st));
  }
  for (int i = 0; i < d.depth; ++i) {
    const long long base = static_cast<long long>(i) * 6 * H;
    FMT_OK(launch_lnmod<T>(h, g, table_e, base + 0, base + H, st));
    FMT_OK(ModeOps<T>::gemm(h, h->A1.p, H, h->qkv[i], epi(EPI_STORE, R, 3 * H, h->qkv[i].b, h->QKV.p, 3 * H, qkv_f32), ks, st));
    FMT_OK(launch_attn<T>(h, g, st));
    {
      EpiParams ep = epi(EPI_GATE_RES, R, H, h->proj[i].b, h->X.p, H, 1);
      ep.gate = table_e; ep.urow = r.urow; ep.ldg = h->NT; ep.gate_off = base + 2 * H;
      FMT_OK(ModeOps<T>::gemm(h, h->A2.p, H, h->proj[i], ep, ks, st));
    }
    FMT_OK(launch_lnmod<T>(h, g, table_e, base + 3 * H, base + 4 * H, st));
    FMT_OK(ModeOps<T>::gemm(h, h->A1.p, H, h->fc1[i], epi(EPI_GELU, R, d.mlp_hidden, h->fc1[i].b, h->Hm.p, d.mlp_hidden, 0), ks, st));
    {
      EpiParams ep = epi(EPI_GATE_RES, R, H, h->fc2[i].b, h->X.p, H, 1);
      ep.gate = table_e; ep.urow = r.urow; ep.ldg = h->NT; ep.gate_off = base + 5 * H;
      FMT_OK(ModeOps<T>::gemm(h, h->Hm.p, d.mlp_hidden, h->fc2[i], ep, ks, st));
    }
  }
  const long long dbase = static_cast<long long>(d.depth) * 6 * H;
  FMT_OK(launch_lnmod<T>(h, g, table_e, dbase, dbase + H, st));
  FMT_OK(ModeOps<T>::gemm(h, h->A1.p, H, h->dec, epi(EPI_STORE, R, s.W, h->dec.b, h->V.p, s.W, 1), ks, st));
  return 0;
}

template <typename T>
static int launch_combine(FmtHandle* h, const ModelShape& s, int mode, float* dst, const float* dt_ptr, cudaStream_t st) {
  const size_t n = static_cast<size_t>(s.B) * s.N * s.W;
  return launch(h, cfg_combine_kernel<T>, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, 1,
                static_cast<const WindowArgs*>(h->wargs.p), s, static_cast<const float*>(h->V.p), mode, dst, dt_ptr, static_cast<T*>(h->ax.p));
}

// ------------------------------------------------------------------------------------------------ persistent window kernel
static bool window_eligible(const FmtHandle* h, const FmtPlan* p) {
  const FmtDims& d = h->d;
  const int R = p->n_branches * p->batch * (d.num_prev_frames + d.frames_per_clip);
  const int nv = d.dim_h / 128;
  return h->use_window != 0 && p->mode == FMT_MODE_BF16 && R <= 256 && p->n_steps * p->n_stages >= 1 && d.depth <= WIN_MAX_DEPTH &&
         (nv == 1 || nv == 2 || nv == 4 || nv == 8) && d.mlp_hidden % 64 == 0 && d.dim_w % 64 == 0;
}

// Builds the device-side description of the window kernel: tensor maps, GEMM item plan, pointers.  Called by fmt_configure
// after the workspace exists.
static int setup_window(FmtHandle* h, cudaStream_t st) {
  const ModelShape& s = h->shape;
  const FmtDims& d = h->d;
  const int R = h->R, H = s.H, M4 = d.mlp_hidden, W = s.W, D = d.depth;
  int Rp = R <= 64 ? 64 : R <= 128 ? 128 : R <= 192 ? 192 : 256;
  const int n_gemms = 2 + 4 * D;
  const int grid = h->num_sms;
  WinParams wp{};
  // grouped schedule: groups of whole sequences (<= 128 rows each), one slice of the SMs per group
  const int n_seq = s.nb * s.B;
  int spg = h->win_spg >= 1 ? h->win_spg : 1;
  if (n_seq % spg != 0 || spg * s.N > 128) spg = 1;
  const bool grouped = h->use_window == 2 && s.N * spg <= 128 && H % 16 == 0 && M4 % 16 == 0 && W % 16 == 0 && grid / (n_seq / spg) >= 8;
  h->win_grouped = grouped;
  if (grouped) {
    wp.G = n_seq / spg; wp.Cg = grid / wp.G; wp.Rg = spg * s.N; wp.RgP = wp.Rg <= 64 ? 64 : 128;
    Rp = wp.G * wp.RgP;                                   // G pre-tiled buffers of RgP rows each
  }
  wp.s = s; wp.R = R; wp.Rp = Rp; wp.depth = D; wp.heads = d.num_heads; wp.window = d.attention_window; wp.mlp_hidden = M4; wp.NT = h->NT;
  wp.n_steps = h->plan.n_steps; wp.n_stages = h->plan.n_stages; wp.n_gemms = n_gemms;

  // accumulator arena: [Pacc (R,H) | QKVacc (R,3H) | Hacc (R,M4) | Vacc (R,W)] fp32, zeroed by one memset per window
  const size_t n_p = static_cast<size_t>(R) * H, n_q = static_cast<size_t>(R) * 3 * H, n_h = static_cast<size_t>(R) * M4, n_v = static_cast<size_t>(R) * W;
  FMT_OK(dev_alloc(h, h->win_acc, (n_p + n_q + n_h + n_v) * 4));
  FMT_OK(dev_alloc(h, h->win_bar, 2048));                 // [0]: grid barrier, [32 * (1 + g)]: barrier of group g (one 128-byte line each)
  FMT_OK(dev_alloc(h, h->win_params, sizeof(WinParams)));
  const int n_maps = n_gemms + 8;
  FMT_OK(dev_alloc(h, h->win_tmaps, static_cast<size_t>(n_maps) * sizeof(CUtensorMap)));
  if (!h->win_err_host) {
    CUDA_OK(cudaHostAlloc(reinterpret_cast<void**>(&h->win_err_host), sizeof(int), cudaHostAllocMapped));
    *h->win_err_host = 0;
    CUDA_OK(cudaHostGetDevicePointer(reinterpret_cast<void**>(&h->win_err_dev), h->win_err_host, 0));
  }
  float* arena = static_cast<float*>(h->win_acc.p);
  wp.Pacc = arena; wp.QKVacc = arena + n_p; wp.Hacc = wp.QKVacc + n_q; wp.Vacc = wp.Hacc + n_h;
  wp.X = static_cast<float*>(h->X.p);
  // pre-tiled operands: [K block][Rp][64] bf16 each, zero-filled once (rows >= R are never written)
  const size_t t_a1 = static_cast<size_t>((H + 63) / 64) * Rp * 64, t_hm = static_cast<size_t>((M4 + 63) / 64) * Rp * 64;
  FMT_OK(dev_alloc(h, h->win_act, (2 * t_a1 + t_hm) * sizeof(bf16)));
  CUDA_OK(cudaMemsetAsync(h->win_act.p, 0, h->win_act.bytes, st));
  wp.A1 = static_cast<bf16*>(h->win_act.p); wp.A2 = wp.A1 + t_a1; wp.Hm = wp.A2 + t_a1; wp.ax = static_cast<bf16*>(h->ax.p);
  wp.table = static_cast<const bf16*>(h->table.p);
  wp.b_x = h->x_emb.b; wp.pos = h->pos; wp.b_dec = h->dec.b;
  for (int i = 0; i < D; ++i) { wp.b_qkv[i] = h->qkv[i].b; wp.b_proj[i] = h->proj[i].b; wp.b_fc1[i] = h->fc1[i].b; wp.b_fc2[i] = h->fc2[i].b; }
  wp.x_state = static_cast<float*>(h->xstate.p); wp.kbuf = static_cast<float*>(h->kbuf.p); wp.ddt = static_cast<const float*>(h->ddt.p);
  for (int i = 0; i < h->plan.n_stages * h->plan.n_stages; ++i) wp.rk_a[i] = h->rk_a[i];
  for (int i = 0; i < h->plan.n_stages; ++i) wp.rk_b[i] = h->rk_b[i];
  wp.wargs = static_cast<const WindowArgs*>(h->wargs.p);
  wp.bar_counter = static_cast<unsigned*>(h->win_bar.p);
  wp.err_flag = h->win_err_dev;
  wp.tmaps = static_cast<const CUtensorMap*>(h->win_tmaps.p);
  wp.w_lookahead = 1000;      // ungated: measured 348 us per ODE step against 378 with a one-stage gate (the gate paid off while spilled state made the SIMT stages' loads slow)
  if (const char* e = getenv("FMT_WIN_LA")) wp.w_lookahead = atoi(e);
  if (getenv("FMT_WIN_TRACE") && atoi(getenv("FMT_WIN_TRACE")) != 0) {
    h->win_trace_stride = h->n_eval * (4 + 8 * D);       // upper bound (the grouped schedule with the fused GELU has 4 + 7 * D stages)
    FMT_OK(dev_alloc(h, h->win_trace, static_cast<size_t>(grid) * h->win_trace_stride * 6 * sizeof(long long)));
    CUDA_OK(cudaMemsetAsync(h->win_trace.p, 0, h->win_trace.bytes, st));
    wp.trace = static_cast<long long*>(h->win_trace.p); wp.trace_stride = h->win_trace_stride;
  }

  std::vector<CUtensorMap> maps(n_maps);
  const int A_AX = n_gemms, A_A1 = n_gemms + 1, A_A2 = n_gemms + 2, A_HM = n_gemms + 3;
  const int C_P = n_gemms + 4, C_Q = n_gemms + 5, C_H = n_gemms + 6, C_V = n_gemms + 7;
  const CUtensorMapDataType BF = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, F32 = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  FMT_OK(make_tmap_ex(h, &maps[A_AX], wp.ax, BF, 2, R, W, W, 64, grouped ? wp.RgP : Rp, CU_TENSOR_MAP_SWIZZLE_128B));
  maps[A_A1] = maps[A_AX]; maps[A_A2] = maps[A_AX]; maps[A_HM] = maps[A_AX];   // A1 / A2 / Hm are pre-tiled: fetched with bulk copies, no tensor map
  FMT_OK(make_tmap_ex(h, &maps[C_P], wp.Pacc, F32, 4, R, H, H, 128, 32, CU_TENSOR_MAP_SWIZZLE_NONE));
  FMT_OK(make_tmap_ex(h, &maps[C_Q], wp.QKVacc, F32, 4, R, 3 * H, 3 * H, 128, 32, CU_TENSOR_MAP_SWIZZLE_NONE));
  FMT_OK(make_tmap_ex(h, &maps[C_H], wp.Hacc, F32, 4, R, M4, M4, 128, 32, CU_TENSOR_MAP_SWIZZLE_NONE));
  FMT_OK(make_tmap_ex(h, &maps[C_V], wp.Vacc, F32, 4, R, W, W, 128, 32, CU_TENSOR_MAP_SWIZZLE_NONE));

  int next_off = 0;
  auto plan_gemm = [&](int g, const Linear& L, int tm_a, int tm_acc, int pk_override) -> int {
    WinGemm& G = wp.gemms[g];
    G.tm_w = g; G.tm_a = tm_a; G.tm_acc = tm_acc; G.N = L.N;
    G.a_tiled = 0;
    if (tm_a == A_A1 || tm_a == A_A2 || tm_a == A_HM) { G.a_tiled = 1; G.tm_a = tm_a == A_A1 ? 0 : tm_a == A_A2 ? 1 : 2; }
    G.n_ft = (L.N + 127) / 128;
    G.nkb = (L.K + 63) / 64;
    REQUIRE(G.n_ft <= grid, "window kernel: %d feature tiles > %d SMs", G.n_ft, grid);
    int pk = grid / G.n_ft;
    if (pk > G.nkb) pk = G.nkb;
    if (pk_override > 0 && pk_override <= pk) pk = pk_override;
    G.pk = pk;
    G.cta_off = next_off;
    next_off = (next_off + G.n_ft * pk) % grid;
    return make_tmap_ex(h, &maps[g], L.w16, BF, 2, L.N, L.K, L.K, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B);
  };
  // grouped schedule: slice the output features over the CTAs of a group; K is split only where one CTA would otherwise
  // have to pull the whole K = mlp_hidden operand (fc2)
  auto plan_gemm2 = [&](int g, const Linear& L, int tm_a, int out, int pk_override, int nf_override, int epi) -> int {
    WinGemm& G = wp.gemms[g];
    G.tm_w = g; G.tm_a = tm_a; G.tm_acc = 0; G.out = out; G.N = L.N;
    G.a_tiled = 0;
    if (tm_a == A_A1 || tm_a == A_A2 || tm_a == A_HM) { G.a_tiled = 1; G.tm_a = tm_a == A_A1 ? 0 : tm_a == A_A2 ? 1 : 2; }
    G.nkb = (L.K + 63) / 64;
    REQUIRE(L.N % 16 == 0, "window kernel: N = %d is not a multiple of 16", L.N);
    int pk = pk_override > 0 ? pk_override : (L.K >= 3072 ? 3 : 1);
    if (pk > G.nkb) pk = G.nkb;
    if (pk > 8) pk = 8;
    int nf = 0;
    for (;;) {                                            // smallest slice that covers N with Cg / pk CTAs, at most 128 wide
      const int slots = wp.Cg / pk;
      nf = slots > 0 ? ((L.N + slots - 1) / slots + 15) / 16 * 16 : 1 << 30;
      for (int c : {16, 32, 48, 64, 96, 128})                // slice widths that pack a 24 KB ring slot (192 / nf K blocks) without waste
        if (nf <= c) { nf = c; break; }
      if (nf <= 128) break;
      REQUIRE(pk > 1, "window kernel: N = %d does not fit %d CTAs per group", L.N, wp.Cg);
      --pk;
    }
    if (nf_override >= 16 && nf_override <= 128 && nf_override % 16 == 0 && ((L.N + nf_override - 1) / nf_override) * pk <= wp.Cg) nf = nf_override;
    G.nf = nf; G.n_nt = (L.N + nf - 1) / nf; G.pk = pk; G.n_ft = G.n_nt;
    G.epi = (epi == 1 && pk == 1) ? 1 : 0;
    G.cta_off = next_off;
    next_off = (next_off + G.n_nt * pk) % wp.Cg;
    return make_tmap_ex(h, &maps[g], L.w16, BF, 2, L.N, L.K, L.K, 64, nf, CU_TENSOR_MAP_SWIZZLE_128B);
  };
  if (grouped) {
    FMT_OK(plan_gemm2(0, h->x_emb, A_AX, 0, 0, 0, 0));
    for (int i = 0; i < D; ++i) {
      FMT_OK(plan_gemm2(1 + 4 * i, h->qkv[i], A_A1, 1, h->win_pk[0], h->win_nf[0], 0));
      FMT_OK(plan_gemm2(2 + 4 * i, h->proj[i], A_A2, 0, h->win_pk[1], h->win_nf[1], 0));
      FMT_OK(plan_gemm2(3 + 4 * i, h->fc1[i], A_A1, 2, h->win_pk[2], h->win_nf[2], h->win_fuse_gelu));
      FMT_OK(plan_gemm2(4 + 4 * i, h->fc2[i], A_HM, 0, h->win_pk[3], h->win_nf[3], 0));
    }
    FMT_OK(plan_gemm2(1 + 4 * D, h->dec, A_A1, 3, 0, 0, 0));
    wp.fuse_gelu = wp.gemms[3].epi;
  } else {
    FMT_OK(plan_gemm(0, h->x_emb, A_AX, C_P, 0));
    for (int i = 0; i < D; ++i) {
      FMT_OK(plan_gemm(1 + 4 * i, h->qkv[i], A_A1, C_Q, h->win_pk[0]));
      FMT_OK(plan_gemm(2 + 4 * i, h->proj[i], A_A2, C_P, h->win_pk[1]));
      FMT_OK(plan_gemm(3 + 4 * i, h->fc1[i], A_A1, C_H, h->win_pk[2]));
      FMT_OK(plan_gemm(4 + 4 * i, h->fc2[i], A_HM, C_P, h->win_pk[3]));
    }
    FMT_OK(plan_gemm(1 + 4 * D, h->dec, A_A1, C_V, 0));
  }
  CUDA_OK(cudaMemcpyAsync(h->win_tmaps.p, maps.data(), maps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(h->win_params.p, &wp, sizeof(WinParams), cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaStreamSynchronize(st));   // `maps` / `wp` are stack objects
  return 0;
}

template <int NV, bool GROUPED>
static int launch_window_nv(FmtHandle* h, cudaStream_t st) {
  constexpr int SMEM = GROUPED ? WIN2_SMEM_BYTES : WIN_SMEM_BYTES;
  static bool attr_set[64] = {};
  if (!attr_set[h->device & 63]) {
    CUDA_OK(cudaFuncSetAttribute(fmt_window_kernel<NV, GROUPED>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    attr_set[h->device & 63] = true;
  }
  int occ = 0;
  CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fmt_window_kernel<NV, GROUPED>, WIN_THREADS, SMEM));
  REQUIRE(occ >= 1, "window kernel does not fit on an SM (%d B smem)", SMEM);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(h->num_sms); cfg.blockDim = dim3(WIN_THREADS); cfg.dynamicSmemBytes = SMEM; cfg.stream = st;
  cudaLaunchAttribute attrs[1];
  attrs[0].id = cudaLaunchAttributeCooperative;      // all CTAs co-resident: the kernel synchronises across the grid
  attrs[0].val.cooperative = 1;
  cfg.attrs = attrs; cfg.numAttrs = 1;
  CUDA_OK(cudaLaunchKernelEx(&cfg, fmt_window_kernel<NV, GROUPED>, static_cast<const WinParams*>(h->win_params.p)));
  count_launch(h);
  return 0;
}

static int launch_window(FmtHandle* h, cudaStream_t st) {
  CUDA_OK(cudaMemsetAsync(h->win_acc.p, 0, h->win_acc.bytes, st));
  CUDA_OK(cudaMemsetAsync(h->win_bar.p, 0, h->win_bar.bytes, st));
  switch (h->shape.H / 128) {
    case 1: return h->win_grouped ? launch_window_nv<1, true>(h, st) : launch_window_nv<1, false>(h, st);
    case 2: return h->win_grouped ? launch_window_nv<2, true>(h, st) : launch_window_nv<2, false>(h, st);
    case 4: return h->win_grouped ? launch_window_nv<4, true>(h, st) : launch_window_nv<4, false>(h, st);
    case 8: return h->win_grouped ? launch_window_nv<8, true>(h, st) : launch_window_nv<8, false>(h, st);
  }
  return set_err(-1, "window kernel: dim_h %d unsupported", h->shape.H);
}

// ------------------------------------------------------------------------------------------------ dataflow window kernel (flow.cuh)
static bool flow_eligible(const FmtHandle* h, const FmtPlan* p) {
  const FmtDims& d = h->d;
  const int N = d.num_prev_frames + d.frames_per_clip;
  const int R = p->n_branches * p->batch * N;
  const int nv = d.dim_h / 128;
  const int CH = h->flow_ch;
  const int nsub = (N + CH - 1) / CH;
  const int hd = d.dim_h / (d.num_heads > 0 ? d.num_heads : 1);
  return h->use_window == 3 && p->mode == FMT_MODE_BF16 && R <= h->flow_max_rows && p->n_steps * p->n_stages >= 1 && d.depth <= WIN_MAX_DEPTH &&
         d.dim_h % 128 == 0 && (nv == 1 || nv == 2 || nv == 4 || nv == 8) && d.mlp_hidden % 64 == 0 && d.dim_w % 64 == 0 &&
         (hd == 32 || hd == 64 || hd == 128) && p->n_branches * p->batch * nsub <= FLOW_MAX_CHUNKS && d.attention_window <= CH &&
         p->n_steps * p->n_stages < 256 && 2 + 4 * d.depth < 256;
}

static int setup_flow(FmtHandle* h, cudaStream_t st) {
  const ModelShape& s = h->shape;
  const FmtDims& d = h->d;
  const int R = h->R, H = s.H, M4 = d.mlp_hidden, W = s.W, D = d.depth;
  const int n_gemms = 2 + 4 * D;
  const int grid = h->num_sms;
  const int CH = h->flow_ch;
  FlowParams& fp = h->flow_params;
  fp = FlowParams{};
  fp.s = s; fp.R = R; fp.depth = D; fp.heads = d.num_heads; fp.window = d.attention_window; fp.mlp_hidden = M4; fp.NT = h->NT;
  fp.n_steps = h->plan.n_steps; fp.n_stages = h->plan.n_stages; fp.n_gemms = n_gemms;
  fp.CH = CH; fp.nsub = (s.N + CH - 1) / CH; fp.NPs = fp.nsub * CH; fp.n_chunks = s.nb * s.B * fp.nsub; fp.RP = fp.n_chunks * CH;
  fp.n_tslots = 512 / CH;
  fp.poll_mode = h->flow_poll;
  fp.fx_c = h->flow_fixed > 0 ? 12582912.f / static_cast<float>(1u << h->flow_fixed) : 0.f;   // 1.5 * 2^23 * 2^-k
  fp.spin_limit = h->flow_spin_limit;
  const size_t RP = fp.RP;

  // fp32 arena, zeroed before every launch: X | Pacc | QKVacc x 2 | Hacc | Vacc, padded rows
  const size_t n_x = RP * H, n_q = RP * 3 * H, n_h = RP * M4, n_v = RP * W;
  FMT_OK(dev_alloc(h, h->flow_acc, (2 * n_x + 2 * n_q + n_h + n_v) * 4));
  float* arena = static_cast<float*>(h->flow_acc.p);
  fp.X = arena; fp.Pacc = fp.X + n_x; fp.QKVacc = fp.Pacc + n_x; fp.Hacc = fp.QKVacc + 2 * n_q; fp.Vacc = fp.Hacc + n_h;
  // pre-tiled operands [chunk][K block][CH][64] bf16, zero-filled once (rows past a chunk's valid rows are never written)
  const size_t t_a1 = static_cast<size_t>(fp.n_chunks) * (H / 64) * CH * 64, t_hm = static_cast<size_t>(fp.n_chunks) * (M4 / 64) * CH * 64;
  FMT_OK(dev_alloc(h, h->flow_act, (2 * t_a1 + t_hm) * sizeof(bf16)));
  CUDA_OK(cudaMemsetAsync(h->flow_act.p, 0, h->flow_act.bytes, st));
  fp.A1 = static_cast<bf16*>(h->flow_act.p); fp.A2 = fp.A1 + t_a1; fp.Hm = fp.A2 + t_a1; fp.ax = static_cast<bf16*>(h->ax.p);
  fp.table = static_cast<const bf16*>(h->table.p);
  fp.U = h->U; fp.urow = h->dedup ? static_cast<const int*>(h->urow_buf.p) : nullptr;
  fp.b_x = h->x_emb.b; fp.pos = h->pos; fp.b_dec = h->dec.b;
  for (int i = 0; i < D; ++i) { fp.b_qkv[i] = h->qkv[i].b; fp.b_proj[i] = h->proj[i].b; fp.b_fc1[i] = h->fc1[i].b; fp.b_fc2[i] = h->fc2[i].b; }
  fp.x_state = static_cast<float*>(h->xstate.p); fp.kbuf = static_cast<float*>(h->kbuf.p); fp.ddt = static_cast<const float*>(h->ddt.p);
  for (int i = 0; i < h->plan.n_stages * h->plan.n_stages; ++i) fp.rk_a[i] = h->rk_a[i];
  for (int i = 0; i < h->plan.n_stages; ++i) fp.rk_b[i] = h->rk_b[i];
  fp.wargs = static_cast<const WindowArgs*>(h->wargs.p);
  // release counters: [n_eval][n_gemms][n_chunks] for the GEMM engine and the same for the SIMT engine
  const size_t n_flags = static_cast<size_t>(h->n_eval) * n_gemms * fp.n_chunks * FLOW_FLAG_STRIDE;
  FMT_OK(dev_alloc(h, h->flow_flags, (2 * n_flags + 2 * FLOW_FLAG_STRIDE) * sizeof(unsigned)));   // + the two rendezvous counters of the trace mode
  fp.g_done = static_cast<unsigned*>(h->flow_flags.p); fp.s_done = fp.g_done + n_flags;
  if (!h->win_err_host) {
    CUDA_OK(cudaHostAlloc(reinterpret_cast<void**>(&h->win_err_host), sizeof(int), cudaHostAllocMapped));
    *h->win_err_host = 0;
    CUDA_OK(cudaHostGetDevicePointer(reinterpret_cast<void**>(&h->win_err_dev), h->win_err_host, 0));
  }
  fp.err_flag = h->win_err_dev;
  fp.trace = nullptr; fp.trace_eval = -1;
  if (getenv("FMT_WIN_TRACE") && atoi(getenv("FMT_WIN_TRACE")) != 0) {
    FMT_OK(dev_alloc(h, h->flow_trace, (static_cast<size_t>(grid) * 2 * n_gemms * fp.n_chunks * 8 + static_cast<size_t>(grid) * 4) * sizeof(long long)));
    CUDA_OK(cudaMemsetAsync(h->flow_trace.p, 0, h->flow_trace.bytes, st));
    fp.trace = static_cast<long long*>(h->flow_trace.p);
    fp.trace_eval = h->n_eval / 2;
    if (const char* e = getenv("FMT_WIN_TRACE_EVAL")) fp.trace_eval = atoi(e);
  }

  // tensor maps: one per GEMM (weights) + ax + accumulators (Pacc, QKVacc parity 0 / 1, Hacc, Vacc)
  const int TM_AX = n_gemms, C_P = n_gemms + 1, C_Q = n_gemms + 2, C_H = n_gemms + 4, C_V = n_gemms + 5, n_maps = n_gemms + 6;
  std::vector<CUtensorMap> maps(n_maps);
  std::vector<FlowGemm> gemms(n_gemms);
  const CUtensorMapDataType BF = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, F32 = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  FMT_OK(make_tmap_ex(h, &maps[TM_AX], fp.ax, BF, 2, R, W, W, 64, CH, CU_TENSOR_MAP_SWIZZLE_128B));
  FMT_OK(make_tmap_ex(h, &maps[C_P], fp.Pacc, F32, 4, fp.RP, H, H, 128, 32, CU_TENSOR_MAP_SWIZZLE_NONE));
  FMT_OK(make_tmap_ex(h, &maps[C_Q], fp.QKVacc, F32, 4, fp.RP, 3 * H, 3 * H, 128, 32, CU_TENSOR_MAP_SWIZZLE_NONE));
  FMT_OK(make_tmap_ex(h, &maps[C_Q + 1], fp.QKVacc + n_q, F32, 4, fp.RP, 3 * H, 3 * H, 128, 32, CU_TENSOR_MAP_SWIZZLE_NONE));
  FMT_OK(make_tmap_ex(h, &maps[C_H], fp.Hacc, F32, 4, fp.RP, M4, M4, 128, 32, CU_TENSOR_MAP_SWIZZLE_NONE));
  FMT_OK(make_tmap_ex(h, &maps[C_V], fp.Vacc, F32, 4, fp.RP, W, W, 128, 32, CU_TENSOR_MAP_SWIZZLE_NONE));
  fp.tm_ax = TM_AX;

  int next_off = 0, max_nk = 1;
  auto plan_gemm = [&](int g, const Linear& L, int a_src, int tm_acc, int pk_override, int par_blk) -> int {
    FlowGemm& G = gemms[g];
    G.tm_w = g; G.tm_acc = tm_acc; G.a_src = a_src; G.par_blk = par_blk;
    G.n_ft = (L.N + 127) / 128;
    G.nkb = (L.K + 63) / 64;
    REQUIRE(G.n_ft <= grid, "flow kernel: %d feature tiles > %d SMs", G.n_ft, grid);
    int pk = grid / G.n_ft;
    if (pk > G.nkb) pk = G.nkb;
    if (pk_override > 0 && pk_override <= pk) pk = pk_override;
    while ((G.nkb + pk - 1) / pk > FLOW_MAX_NW - 1 && pk < G.nkb) ++pk;      // an item's weight tiles must fit the ring
    REQUIRE((G.nkb + pk - 1) / pk <= FLOW_MAX_NW - 1 && G.n_ft * pk <= grid, "flow kernel: K = %d does not fit the weight ring", L.K);
    G.pk = pk;
    G.n_items = G.n_ft * pk;
    G.cta_off = next_off;
    next_off = (next_off + G.n_items) % grid;
    const int nk = (G.nkb + pk - 1) / pk;
    if (nk > max_nk) max_nk = nk;
    return make_tmap_ex(h, &maps[g], L.w16, BF, 2, L.N, L.K, L.K, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B);
  };
  FMT_OK(plan_gemm(0, h->x_emb, 0, C_P, 0, -1));
  for (int i = 0; i < D; ++i) {
    FMT_OK(plan_gemm(1 + 4 * i, h->qkv[i], 1, C_Q, h->win_pk[0], i));
    FMT_OK(plan_gemm(2 + 4 * i, h->proj[i], 2, C_P, h->win_pk[1], -1));
    FMT_OK(plan_gemm(3 + 4 * i, h->fc1[i], 1, C_H, h->win_pk[2], -1));
    FMT_OK(plan_gemm(4 + 4 * i, h->fc2[i], 3, C_P, h->win_pk[3], -1));
  }
  FMT_OK(plan_gemm(1 + 4 * D, h->dec, 1, C_V, 0, -1));
  // shared memory: 2 staging tiles + activation ring (slots of the largest item's K range) + weight ring with what is left
  fp.a_slot_bytes = max_nk * CH * 128;
  fp.na = CH <= 32 ? 3 : 2;
  if (const char* e = getenv("FMT_FLOW_NA")) { const int v = atoi(e); if (v >= 2 && v <= FLOW_MAX_NA) fp.na = v; }
  const int left = FLOW_SMEM_MAX - 1024 - FLOW_BAR_BYTES - 2 * FLOW_STG_BYTES - fp.na * fp.a_slot_bytes;
  fp.nw = left / FLOW_W_BYTES;
  if (fp.nw > FLOW_MAX_NW) fp.nw = FLOW_MAX_NW;
  if (const char* e = getenv("FMT_FLOW_NW")) { const int v = atoi(e); if (v >= 2 && v <= fp.nw) fp.nw = v; }
  REQUIRE(fp.nw >= max_nk + 1, "flow kernel: weight ring of %d slots cannot hold an item of %d K blocks", fp.nw, max_nk);

  FMT_OK(dev_alloc(h, h->flow_gemms, gemms.size() * sizeof(FlowGemm)));
  FMT_OK(dev_alloc(h, h->flow_tmaps, maps.size() * sizeof(CUtensorMap)));
  CUDA_OK(cudaMemcpyAsync(h->flow_gemms.p, gemms.data(), gemms.size() * sizeof(FlowGemm), cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(h->flow_tmaps.p, maps.data(), maps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaStreamSynchronize(st));   // `maps` / `gemms` are stack objects
  fp.gemms = static_cast<const FlowGemm*>(h->flow_gemms.p);
  fp.tmaps = static_cast<const CUtensorMap*>(h->flow_tmaps.p);
  return 0;
}

static int flow_smem_bytes(const FlowParams& fp) {
  return 1024 + fp.nw * FLOW_W_BYTES + fp.na * fp.a_slot_bytes + 2 * FLOW_STG_BYTES + FLOW_BAR_BYTES;
}

template <int NV>
static int launch_flow_nv(FmtHandle* h, cudaStream_t st, bool probe_only) {
  const int smem = flow_smem_bytes(h->flow_params);
  CUDA_OK(cudaFuncSetAttribute(fmt_flow_kernel<NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  int occ = 0;
  CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fmt_flow_kernel<NV>, FLOW_THREADS, smem));
  REQUIRE(occ >= 1, "flow kernel does not fit on an SM (%d B smem)", smem);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(h->num_sms); cfg.blockDim = dim3(FLOW_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attrs[1];
  attrs[0].id = cudaLaunchAttributeCooperative;      // all CTAs co-resident: they wait for one another's counters
  attrs[0].val.cooperative = 1;
  cfg.attrs = attrs; cfg.numAttrs = 1;
  if (probe_only) {
    // one trial launch with zero evaluations (every role loop is empty): under MPS with an SM limit, a green context or any other
    // reason the runtime cannot make num_sms CTAs co-resident, THIS is where it says so - and the plan runs one kernel per op instead
    FlowParams trial = h->flow_params;
    trial.n_steps = 0; trial.trace = nullptr;
    CUDA_OK(cudaLaunchKernelEx(&cfg, fmt_flow_kernel<NV>, trial));
    CUDA_OK(cudaStreamSynchronize(st));
    return 0;
  }
  CUDA_OK(cudaLaunchKernelEx(&cfg, fmt_flow_kernel<NV>, h->flow_params));
  count_launch(h);
  return 0;
}

static int launch_flow(FmtHandle* h, cudaStream_t st, bool probe_only = false) {
  if (!probe_only) {
    CUDA_OK(cudaMemsetAsync(h->flow_acc.p, 0, h->flow_acc.bytes, st));
    CUDA_OK(cudaMemsetAsync(h->flow_flags.p, 0, h->flow_flags.bytes, st));
  }
  switch (h->shape.H / 128) {
    case 1: return launch_flow_nv<1>(h, st, probe_only);
    case 2: return launch_flow_nv<2>(h, st, probe_only);
    case 4: return launch_flow_nv<4>(h, st, probe_only);
    case 8: return launch_flow_nv<8>(h, st, probe_only);
  }
  return set_err(-1, "flow kernel: dim_h %d unsupported", h->shape.H);
}

// The whole window: prepare -> tables -> S steps x stages -> finalize.  This is what gets captured in the graph.
template <typename T>
static int enqueue_window(FmtHandle* h, const GraphShape& gs, cudaStream_t st) {
  const ModelShape& s = gs.s;
  const WindowArgs* wa = static_cast<const WindowArgs*>(h->wargs.p);
  const size_t nx = static_cast<size_t>(s.B) * s.L * s.W, nfull = static_cast<size_t>(s.B) * s.N * s.W;
  float* x_state = static_cast<float*>(h->xstate.p);
  float* y_stage = static_cast<float*>(h->ystage.p);
  float* kbuf = static_cast<float*>(h->kbuf.p);
  T* ax = static_cast<T*>(h->ax.p);
  const float* ddt = static_cast<const float*>(h->ddt.p);
  const int S = h->plan.n_steps, G = h->plan.n_stages;
  const dim3 gx(static_cast<unsigned>((nx + 255) / 256)), blk(256);
  const int chunk = gs.rows.chunk;

  FMT_OK(launch(h, init_window_kernel<T>, dim3(static_cast<unsigned>((nfull + 255) / 256)), blk, 0, st, 1, wa, s, x_state,
                static_cast<float*>(h->prevx.p), ax));
  if (S > 0) FMT_OK(enqueue_prepare<T>(h, gs, st));
  if (h->window_active && S > 0) {
    // small-R plan: every evaluation of the window runs inside ONE persistent kernel (flow.cuh; window.cuh with FMT_WINDOW=1/2)
    FMT_OK(enqueue_tables<T>(h, gs, 0, h->n_eval, st));
    if (h->flow_active) FMT_OK(launch_flow(h, st));
    else FMT_OK(launch_window(h, st));
    FMT_OK(launch(h, finalize_window_kernel, gx, blk, 0, st, 1, wa, s, static_cast<const float*>(x_state), static_cast<float*>(h->prevx.p)));
    return 0;
  }
  for (int step = 0; step < S; ++step) {
    for (int g = 0; g < G; ++g) {
      const int e = step * G + g;
      if (e % chunk == 0) {
        const int n = (h->n_eval - e) < chunk ? (h->n_eval - e) : chunk;
        FMT_OK(enqueue_tables<T>(h, gs, e, n, st));
      }
      if (g > 0) {   // y_g = y0 + dt * sum_j a[g][j] k_j  (also refreshes the x-embedder operand)
        const float* a = &h->rk_a[g * G];
        FMT_OK(launch(h, rk_combine_kernel<T>, gx, blk, 0, st, 1, s, static_cast<const float*>(x_state), y_stage, static_cast<const float*>(kbuf), nx, nx, g,
                      a[0], G > 1 ? a[1] : 0.f, G > 2 ? a[2] : 0.f, G > 3 ? a[3] : 0.f, ddt + step, ax));
      }
      FMT_OK(enqueue_forward<T>(h, gs, e % chunk, st));
      if (G == 1) FMT_OK(launch_combine<T>(h, s, 2, x_state, ddt + step, st));           // fused CFG + Euler
      else FMT_OK(launch_combine<T>(h, s, 1, kbuf + static_cast<size_t>(g) * nx, nullptr, st));
    }
    if (G > 1) {
      const float* b = h->rk_b.data();
      FMT_OK(launch(h, rk_combine_kernel<T>, gx, blk, 0, st, 1, s, static_cast<const float*>(x_state), x_state, static_cast<const float*>(kbuf), nx, nx, G,
                    b[0], G > 1 ? b[1] : 0.f, G > 2 ? b[2] : 0.f, G > 3 ? b[3] : 0.f, ddt + step, ax));
    }
  }
  FMT_OK(launch(h, finalize_window_kernel, gx, blk, 0, st, 1, wa, s, static_cast<const float*>(x_state), static_cast<float*>(h->prevx.p)));
  return 0;
}

static int enqueue_window_mode(FmtHandle* h, const GraphShape& gs, cudaStream_t st) {
  switch (h->plan.mode) {
    case FMT_MODE_BF16: return enqueue_window<bf16>(h, gs, st);
    case FMT_MODE_BF16X3: return enqueue_window<bf16x3_t>(h, gs, st);
  }
  return enqueue_window<float>(h, gs, st);
}

// The per-slot window graph: the plan's evaluation count, every slot on its own schedule (SlotOde), always one kernel per op.  Each
// evaluation e is [the stage combine of the slots at a stage > 0 (e > 0)] -> forward -> [CFG combine + the ODE update of each slot
// that is at an evaluation of its own].
template <typename T>
static int enqueue_window_ode(FmtHandle* h, const GraphShape& gs, cudaStream_t st) {
  const ModelShape& s = gs.s;
  const WindowArgs* wa = static_cast<const WindowArgs*>(h->wargs.p);
  const size_t nx = static_cast<size_t>(s.B) * s.L * s.W, nfull = static_cast<size_t>(s.B) * s.N * s.W;
  float* x_state = static_cast<float*>(h->xstate.p);
  float* kbuf = static_cast<float*>(h->s_kbuf.p);
  T* ax = static_cast<T*>(h->ax.p);
  const dim3 gx(static_cast<unsigned>((nx + 255) / 256)), gfull(static_cast<unsigned>((nfull + 255) / 256)), blk(256);
  const CondRows& r = gs.rows;
  const int ne = h->n_eval;

  FMT_OK(launch(h, init_window_kernel<T>, gfull, blk, 0, st, 1, wa, s, x_state, static_cast<float*>(h->prevx.p), ax));
  if (ne > 0) FMT_OK(enqueue_prepare<T>(h, gs, st));
  for (int e = 0; e < ne; ++e) {
    if (e % r.chunk == 0) FMT_OK(enqueue_tables<T>(h, gs, e, std::min(ne - e, r.chunk), st));
    if (e > 0)
      FMT_OK(launch(h, sched_stage_kernel<T>, gx, blk, 0, st, 1, wa, s, static_cast<const float*>(x_state), static_cast<float*>(h->ystage.p),
                    static_cast<const float*>(kbuf), nx, e, ax));
    FMT_OK(enqueue_forward<T>(h, gs, e % r.chunk, st));
    FMT_OK(launch(h, sched_combine_kernel<T>, gfull, blk, 0, st, 1, wa, s, static_cast<const float*>(h->V.p), e, x_state, kbuf, nx, ax));
  }
  FMT_OK(launch(h, finalize_window_kernel, gx, blk, 0, st, 1, wa, s, static_cast<const float*>(x_state), static_cast<float*>(h->prevx.p)));
  return 0;
}

static int enqueue_window_ode_mode(FmtHandle* h, const GraphShape& gs, cudaStream_t st) {
  switch (h->plan.mode) {
    case FMT_MODE_BF16: return enqueue_window_ode<bf16>(h, gs, st);
    case FMT_MODE_BF16X3: return enqueue_window_ode<bf16x3_t>(h, gs, st);
  }
  return enqueue_window_ode<float>(h, gs, st);
}

// Destroys the occupancy buckets' graphs and maps (the caller has synchronised the stream that replays them)
static void drop_buckets(FmtHandle* h) {
  for (FmtHandle::Bucket& b : h->buckets) {
    if (b.exec) cudaGraphExecDestroy(b.exec);
    if (b.ode_exec) cudaGraphExecDestroy(b.ode_exec);
    if (b.s_map.p) { cudaFree(b.s_map.p); h->ws_bytes -= b.s_map.bytes; }
  }
  h->buckets.clear();
}

// Captures one window of enqueue(h, gs, .) as a CUDA graph; *launches: the kernels it holds (counted by launch())
static int capture_window(FmtHandle* h, int (*enqueue)(FmtHandle*, const GraphShape&, cudaStream_t), const GraphShape& gs, cudaGraphExec_t* exec,
                          int* nodes, long long* launches) {
  cudaGraph_t graph = nullptr;
  cudaStream_t cs;
  CUDA_OK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
  // make sure the lazily-set function attributes exist before capture (attribute calls are not capturable work but are legal)
  CUDA_OK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
  const long long outer = h->capture_launches;
  h->capturing = true; h->capture_launches = 0;
  int rc = enqueue(h, gs, cs);
  h->capturing = false;
  const long long counted = h->capture_launches;
  h->capture_launches = outer;
  cudaError_t ce = cudaStreamEndCapture(cs, &graph);
  if (rc != 0) { if (graph) cudaGraphDestroy(graph); cudaStreamDestroy(cs); return rc; }
  if (ce != cudaSuccess) { cudaStreamDestroy(cs); return set_err(-2, "graph capture failed: %s", cudaGetErrorString(ce)); }
  size_t n_nodes = 0;
  cudaGraphGetNodes(graph, nullptr, &n_nodes);
  *nodes = static_cast<int>(n_nodes);
  ce = cudaGraphInstantiate(exec, graph, 0);
  cudaGraphDestroy(graph);
  cudaStreamDestroy(cs);
  if (ce != cudaSuccess) return set_err(-2, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ce));
  *launches = counted;
  return 0;
}

// ------------------------------------------------------------------------------------------------ create / destroy
static int upload(FmtHandle* h, const void* src, size_t n_floats, int location, float** out) {
  float* p = nullptr;
  CUDA_OK(cudaMalloc(&p, n_floats * sizeof(float)));
  h->owned.push_back(p);
  CUDA_OK(cudaMemcpy(p, src, n_floats * sizeof(float), location == FMT_LOC_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice));
  *out = p;
  return 0;
}

// FMT_MODE_BF16X3 operand of a Linear: (N, 2K) pairs from its fp32 (padded) weight, once per Linear
static int pack_split(FmtHandle* h, Linear& L, cudaStream_t st) {
  if (L.w3) return 0;
  REQUIRE(L.K % 64 == 0, "bf16x3 mode: K = %d is not a multiple of 64", L.K);
  const size_t n = static_cast<size_t>(L.N) * L.K;
  CUDA_OK(cudaMalloc(&L.w3, n * sizeof(bf16x3_t)));
  h->owned.push_back(L.w3);
  f32_to_split_kernel<<<static_cast<unsigned>(std::min<size_t>((n / 4 + 255) / 256, static_cast<size_t>(h->num_sms) * 16)), 256, 0, st>>>(
      L.w32, reinterpret_cast<bf16x3_t*>(L.w3), n / 4);
  LAUNCH_CHECK();
  return 0;
}

static int pack_split_all(FmtHandle* h, cudaStream_t st) {
  for (Linear* L : {&h->x_emb, &h->c_emb, &h->ada, &h->dec}) FMT_OK(pack_split(h, *L, st));
  for (int i = 0; i < h->d.depth; ++i)
    for (Linear* L : {&h->qkv[i], &h->proj[i], &h->fc1[i], &h->fc2[i]}) FMT_OK(pack_split(h, *L, st));
  return 0;
}

static int make_linear(FmtHandle* h, Linear& L, const void* w, const void* b, int N, int K, int Kpad, int location) {
  float *w_raw = nullptr;
  FMT_OK(upload(h, w, static_cast<size_t>(N) * K, location, &w_raw));
  FMT_OK(upload(h, b, N, location, &L.b));
  L.N = N; L.K = Kpad;
  const size_t n = static_cast<size_t>(N) * Kpad;
  CUDA_OK(cudaMalloc(&L.w16, n * sizeof(bf16)));
  h->owned.push_back(L.w16);
  pack_weight_kernel<<<static_cast<unsigned>((n + 255) / 256), 256>>>(w_raw, N, K, L.w16, Kpad);
  LAUNCH_CHECK();
  if (Kpad == K) {
    L.w32 = w_raw;
  } else {
    CUDA_OK(cudaMalloc(&L.w32, n * sizeof(float)));
    h->owned.push_back(L.w32);
    pad_weight_f32_kernel<<<static_cast<unsigned>((n + 255) / 256), 256>>>(w_raw, N, K, L.w32, Kpad);
    LAUNCH_CHECK();
  }
  return 0;
}

static int debug_handle(FmtHandle& h) {
  int dev = 0;
  CUDA_OK(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return set_err(-4, "device is sm_%d%d; sm_100a required", prop.major, prop.minor);
  h.device = dev; h.num_sms = prop.multiProcessorCount;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  CUDA_OK(cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &fn, 12000, cudaEnableDefault, &qres));
  REQUIRE(fn && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
  h.encode = reinterpret_cast<PFN_encodeTiled>(fn);
  return 0;
}

extern "C" {

int32_t fmt_abi_version(void) { return FMT_ABI_VERSION; }
const char* fmt_last_error(void) { return g_err; }

int32_t fmt_create(const FmtDims* dims, const void* const* wp, int32_t n_ptrs, int32_t location, int32_t device, FmtHandle** out) {
  REQUIRE(dims && wp && out, "fmt_create: null argument");
  const FmtDims& d = *dims;
  REQUIRE(n_ptrs == FMT_W_NUM_GLOBAL + d.depth * FMT_W_PER_BLOCK, "fmt_create: expected %d weight pointers, got %d",
          FMT_W_NUM_GLOBAL + d.depth * FMT_W_PER_BLOCK, n_ptrs);
  for (int i = 0; i < n_ptrs; ++i) REQUIRE(wp[i] != nullptr, "fmt_create: weight pointer %d is null", i);
  REQUIRE(d.dim_h % 128 == 0 && d.dim_w % 64 == 0 && d.dim_a % 4 == 0 && d.mlp_hidden % 64 == 0,
          "fmt_create: unsupported dims (dim_h %% 128, dim_w %% 64, mlp_hidden %% 64 required)");
  REQUIRE(d.dim_h % d.num_heads == 0, "fmt_create: dim_h must be divisible by num_heads");
  const int hd = d.dim_h / d.num_heads;
  REQUIRE(hd == 32 || hd == 64 || hd == 128, "fmt_create: head_dim %d unsupported (32, 64, 128)", hd);
  REQUIRE(d.num_prev_frames <= d.frames_per_clip && d.num_prev_frames >= 0 && d.frames_per_clip > 0, "fmt_create: need 0 <= P <= L");
  REQUIRE(d.attention_window >= 0, "fmt_create: attention_window must be >= 0");

  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0)
    return set_err(-4, "fmt_create: no CUDA device - this library has no CPU fallback");
  REQUIRE(device >= 0 && device < n_dev, "fmt_create: device %d out of range (%d devices)", device, n_dev);
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return set_err(-4, "fmt_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
  CUDA_OK(cudaSetDevice(device));

  FmtHandle* h = new FmtHandle();
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  h->d = d;
  h->N = d.num_prev_frames + d.frames_per_clip;
  h->Kc = ((d.dim_w + d.dim_a + d.dim_e + 63) / 64) * 64;
  h->NT = d.depth * 6 * d.dim_h + 2 * d.dim_h;
  if (const char* e = getenv("FMT_PDL")) h->use_pdl = atoi(e) != 0;
  if (const char* e = getenv("FMT_WINDOW")) h->use_window = atoi(e);
  if (const char* e = getenv("FMT_FLOW_CH")) { const int v = atoi(e); if (v == 32 || v == 64) h->flow_ch = v; }
  if (const char* e = getenv("FMT_FLOW_MAX_ROWS")) h->flow_max_rows = atoi(e);
  if (const char* e = getenv("FMT_FLOW_POLL")) h->flow_poll = atoi(e);
  if (const char* e = getenv("FMT_DEDUP")) h->use_dedup = atoi(e) != 0;
  if (const char* e = getenv("FMT_FLOW_FIXED")) { const int v = atoi(e); if (v >= 0 && v <= 22) h->flow_fixed = v; }
  if (const char* e = getenv("FMT_FLOW_SPIN_MS")) h->flow_spin_limit = static_cast<long long>(atof(e) * 1.9e6);
  if (const char* e = getenv("FMT_WIN_SPG")) h->win_spg = atoi(e);
  if (const char* e = getenv("FMT_WIN_FUSE_GELU")) h->win_fuse_gelu = atoi(e) != 0;
  if (const char* e = getenv("FMT_WIN_NF")) sscanf(e, "%d,%d,%d,%d", &h->win_nf[0], &h->win_nf[1], &h->win_nf[2], &h->win_nf[3]);
  if (const char* e = getenv("FMT_PAIR")) h->use_pair = atoi(e) != 0;
  if (const char* e = getenv("FMT_SPLITK")) h->use_splitk = atoi(e) != 0;
  if (const char* e = getenv("FMT_RASTER_GM")) { int v = atoi(e); if (v >= 1) h->raster_gm = v; }
  if (const char* e = getenv("FMT_WIN_PK")) sscanf(e, "%d,%d,%d,%d", &h->win_pk[0], &h->win_pk[1], &h->win_pk[2], &h->win_pk[3]);
  {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &fn, 12000, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || fn == nullptr) {
      delete h;
      return set_err(-3, "fmt_create: cuTensorMapEncodeTiled not available from the driver");
    }
    h->encode = reinterpret_cast<PFN_encodeTiled>(fn);
  }
  const int H = d.dim_h;
  int rc = 0;
#define TRY(expr) do { rc = (expr); if (rc != 0) { fmt_destroy(h); return rc; } } while (0)
  TRY(make_linear(h, h->x_emb, wp[FMT_W_X_W], wp[FMT_W_X_B], H, d.dim_w, d.dim_w, location));
  TRY(make_linear(h, h->c_emb, wp[FMT_W_C_W], wp[FMT_W_C_B], H, d.dim_w + d.dim_a + d.dim_e, h->Kc, location));
  TRY(make_linear(h, h->dec, wp[FMT_W_DEC_W], wp[FMT_W_DEC_B], d.dim_w, H, H, location));
  TRY(upload(h, wp[FMT_W_T0_W], static_cast<size_t>(H) * 256, location, &h->t0_w));
  TRY(upload(h, wp[FMT_W_T0_B], H, location, &h->t0_b));
  TRY(upload(h, wp[FMT_W_T2_W], static_cast<size_t>(H) * H, location, &h->t2_w));
  TRY(upload(h, wp[FMT_W_T2_B], H, location, &h->t2_b));
  TRY(upload(h, wp[FMT_W_POS], static_cast<size_t>(h->N) * H, location, &h->pos));
  h->qkv.resize(d.depth); h->proj.resize(d.depth); h->fc1.resize(d.depth); h->fc2.resize(d.depth);
  // concatenated AdaLN projection: rows [block0 (6H) | ... | block{depth-1} (6H) | decoder (2H)]
  {
    Linear& A = h->ada;
    A.N = h->NT; A.K = H;
    const size_t n = static_cast<size_t>(h->NT) * H;
    cudaError_t e1 = cudaMalloc(&A.w32, n * sizeof(float));
    cudaError_t e2 = cudaMalloc(&A.w16, n * sizeof(bf16));
    cudaError_t e3 = cudaMalloc(&A.b, static_cast<size_t>(h->NT) * sizeof(float));
    if (A.w32) h->owned.push_back(A.w32);
    if (A.w16) h->owned.push_back(A.w16);
    if (A.b) h->owned.push_back(A.b);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) { fmt_destroy(h); return set_err(-2, "fmt_create: cudaMalloc failed for the AdaLN table weights"); }
  }
  const cudaMemcpyKind kind = location == FMT_LOC_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  for (int i = 0; i < d.depth; ++i) {
    const void* const* bp = wp + FMT_W_NUM_GLOBAL + i * FMT_W_PER_BLOCK;
    TRY(make_linear(h, h->qkv[i], bp[FMT_WB_QKV_W], bp[FMT_WB_QKV_B], 3 * H, H, H, location));
    TRY(make_linear(h, h->proj[i], bp[FMT_WB_PROJ_W], bp[FMT_WB_PROJ_B], H, H, H, location));
    TRY(make_linear(h, h->fc1[i], bp[FMT_WB_FC1_W], bp[FMT_WB_FC1_B], d.mlp_hidden, H, H, location));
    TRY(make_linear(h, h->fc2[i], bp[FMT_WB_FC2_W], bp[FMT_WB_FC2_B], H, d.mlp_hidden, d.mlp_hidden, location));
    if (cudaMemcpy(h->ada.w32 + static_cast<size_t>(i) * 6 * H * H, bp[FMT_WB_ADA_W], static_cast<size_t>(6) * H * H * sizeof(float), kind) != cudaSuccess ||
        cudaMemcpy(h->ada.b + static_cast<size_t>(i) * 6 * H, bp[FMT_WB_ADA_B], static_cast<size_t>(6) * H * sizeof(float), kind) != cudaSuccess) {
      fmt_destroy(h);
      return set_err(-2, "fmt_create: copying adaLN weights of block %d failed", i);
    }
  }
  if (cudaMemcpy(h->ada.w32 + static_cast<size_t>(d.depth) * 6 * H * H, wp[FMT_W_DEC_ADA_W], static_cast<size_t>(2) * H * H * sizeof(float), kind) != cudaSuccess ||
      cudaMemcpy(h->ada.b + static_cast<size_t>(d.depth) * 6 * H, wp[FMT_W_DEC_ADA_B], static_cast<size_t>(2) * H * sizeof(float), kind) != cudaSuccess) {
    fmt_destroy(h);
    return set_err(-2, "fmt_create: copying decoder adaLN weights failed");
  }
  {
    const size_t n = static_cast<size_t>(h->NT) * H;
    pack_weight_kernel<<<static_cast<unsigned>((n + 255) / 256), 256>>>(h->ada.w32, h->NT, H, h->ada.w16, H);
  }
  if (cudaDeviceSynchronize() != cudaSuccess || cudaGetLastError() != cudaSuccess) {
    fmt_destroy(h);
    return set_err(-2, "fmt_create: weight packing failed: %s", cudaGetErrorString(cudaGetLastError()));
  }
#undef TRY
  *out = h;
  return 0;
}

int32_t fmt_destroy(FmtHandle* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
  if (h->ode_exec) cudaGraphExecDestroy(h->ode_exec);
  drop_buckets(h);
  for (void* p : h->owned) cudaFree(p);
  for (auto& kv : h->ode_cache) cudaFree(kv.second.p);
  DevBuf* bufs[] = {&h->cond, &h->cemb, &h->temb, &h->tfreq, &h->th, &h->silu, &h->table, &h->xstate, &h->ystage, &h->kbuf, &h->prevx, &h->ax,
                    &h->X, &h->A1, &h->QKV, &h->A2, &h->Hm, &h->V, &h->ddt, &h->dteval, &h->wargs, &h->st_rs, &h->st_wa, &h->st_we, &h->st_noise, &h->st_rd, &h->ev_wa, &h->ev_we,
                    &h->win_params, &h->win_tmaps, &h->win_acc, &h->win_bar, &h->win_trace, &h->win_act,
                    &h->flow_gemms, &h->flow_tmaps, &h->flow_acc, &h->flow_act, &h->flow_flags, &h->flow_trace, &h->urow_buf, &h->uidx_buf,
                    &h->slot_buf, &h->slot_zero, &h->s_cond, &h->s_cemb, &h->s_urow, &h->s_uidx, &h->s_kbuf, &h->bucket_maps};
  for (DevBuf* b : bufs)
    if (b->p) cudaFree(b->p);
  if (h->win_err_host) cudaFreeHost(h->win_err_host);
  if (h->slot_host) cudaFreeHost(h->slot_host);
  if (h->slot_ev) cudaEventDestroy(h->slot_ev);
  delete h;
  return 0;
}

int64_t fmt_workspace_bytes(const FmtHandle* h) { return h ? static_cast<int64_t>(h->ws_bytes) : 0; }
int64_t fmt_launch_count(const FmtHandle* hc, int32_t reset) {
  FmtHandle* h = const_cast<FmtHandle*>(hc);
  if (!h) return 0;
  const long long v = h->launches;
  if (reset) h->launches = 0;
  return v;
}
int32_t fmt_graph_kernel_nodes(const FmtHandle* h) { return h ? h->graph_nodes : 0; }
int32_t fmt_last_window_slots(const FmtHandle* h) { return h ? h->last_slots : 0; }
int32_t fmt_ode_graph_kernel_nodes(const FmtHandle* h) { return h ? h->ode_nodes : 0; }
int64_t fmt_debug_window_trace(const FmtHandle* h, int64_t* out, int64_t max_elems) {
  if (h && h->flow_active && h->flow_trace.p) {   // dataflow kernel: [cta][engine][stage][chunk][4] SM-clock stamps
    const int64_t nf = static_cast<int64_t>(h->flow_trace.bytes / sizeof(long long));
    if (out != nullptr && max_elems >= nf) {
      if (cudaMemcpy(out, h->flow_trace.p, nf * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    }
    return nf;
  }
  if (!h || !h->win_trace.p) return 0;
  const int64_t n = static_cast<int64_t>(h->num_sms) * h->win_trace_stride * 6;
  if (out != nullptr && max_elems >= n) {
    if (cudaMemcpy(out, h->win_trace.p, n * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  }
  return n;
}
int32_t fmt_window_kernel_status(const FmtHandle* h) {
  if (!h || !h->window_active) return -1;
  const int trapped = h->win_err_host ? *h->win_err_host : 0;
  if (trapped != 0) return trapped;             // a tripped spin of an earlier window stays visible after per-slot calls
  return h->last_ode ? -1 : 0;
}

// Which token rows (branch, clip, frame) see the same condition row [wr | wa | we]?  urow[row] = index of the row's distinct
// condition row, uidx[u] = the first token row that sees distinct row u.  The key is exactly what cond_gather_kernel reads for a
// row: the identity latent unless nulled (per clip), the audio latent (context frames read prev_wa, never nulled, FMT.py:366,388;
// current frames read wa unless nulled), the emotion (nulled; else slot b's mode we_dyn[b]: static = per clip, covering the context
// frames too, FMT.py:325-326; dynamic = per frame).  per_slot: rows of different slots are never shared (the per-slot window graph,
// whose slots have their own times): only the truly-uncond current frames of 4-branch plans, [0 | 0 | 0] in every slot, are affected.
// The map does not depend on we_dyn: in every branch that keeps the emotion (branch_nulls) the audio term is kept too or is a context
// frame's prev_wa, and both are keyed by (clip, frame) already.  So one map serves every mix of static and dynamic slots, and a call
// that mixes them replays the graphs of the plan (fmt_debug_condition_rows_slots shows the map for any mix).
static void distinct_condition_rows(const ModelShape& s, const int32_t* we_dyn, std::vector<int>& urow, std::vector<int>& uidx,
                                    bool per_slot = false) {
  const int R = s.nb * s.B * s.N;
  urow.assign(R, 0);
  uidx.clear();
  std::map<std::tuple<int, int, int, int, int, int, int, int>, int> seen;
  for (int row = 0; row < R; ++row) {
    const int br = row / (s.B * s.N), b = (row / s.N) % s.B, f = row % s.N;
    const bool za = (s.null_a >> br) & 1, zr = (s.null_r >> br) & 1, ze = (s.null_e >> br) & 1, ctx = f < s.P;
    const int kr = zr ? -1 : b;
    const int ka = ctx ? 0 : (za ? 1 : 2), kab = (ctx || !za) ? b : -1, kaf = (ctx || !za) ? f : -1;
    const int ke = ze ? 0 : (we_dyn[b] ? 2 : 1), keb = ze ? -1 : b, kef = (!ze && we_dyn[b]) ? f : -1;
    const auto key = std::make_tuple(kr, ka, kab, kaf, ke, keb, kef, per_slot ? b : -1);
    auto it = seen.find(key);
    if (it == seen.end()) { it = seen.emplace(key, static_cast<int>(uidx.size())).first; uidx.push_back(row); }
    urow[row] = it->second;
  }
}

static void branch_nulls(ModelShape& s) {
  if (s.nb == 3) { s.null_a = 0b001; s.null_r = 0; s.null_e = 0b101; }            // [uncond | all | audio-only]   FMT.py:360-362
  else if (s.nb == 4) { s.null_a = 0b0011; s.null_r = 0b0001; s.null_e = 0b1011; } // [truly-uncond | uncond | all | audio-only] :382-384
  else { s.null_a = s.null_r = s.null_e = 0; }
}

// Host-only view of the deduplication for tests (no device work): fills urow[n_branches * batch * n_frames], returns U.
int32_t fmt_debug_condition_rows(int32_t n_branches, int32_t batch, int32_t n_frames, int32_t n_prev, int32_t we_dynamic, int32_t* urow_out) {
  return fmt_debug_condition_rows_ode(n_branches, batch, n_frames, n_prev, we_dynamic, 0, urow_out);
}

int32_t fmt_debug_condition_rows_ode(int32_t n_branches, int32_t batch, int32_t n_frames, int32_t n_prev, int32_t we_dynamic, int32_t per_slot,
                                     int32_t* urow_out) {
  if (batch < 1) return -1;
  const std::vector<int32_t> modes(batch, we_dynamic);
  return fmt_debug_condition_rows_slots(n_branches, batch, n_frames, n_prev, modes.data(), per_slot, urow_out);
}

int32_t fmt_debug_condition_rows_slots(int32_t n_branches, int32_t batch, int32_t n_frames, int32_t n_prev, const int32_t* we_dynamic,
                                       int32_t per_slot, int32_t* urow_out) {
  if (n_branches < 1 || n_branches > 4 || batch < 1 || n_frames < 1 || n_prev < 0 || n_prev > n_frames || we_dynamic == nullptr) return -1;
  ModelShape s{};
  s.nb = n_branches; s.B = batch; s.N = n_frames; s.P = n_prev;
  branch_nulls(s);
  std::vector<int> urow, uidx;
  distinct_condition_rows(s, we_dynamic, urow, uidx, per_slot != 0);
  if (urow_out != nullptr) std::copy(urow.begin(), urow.end(), urow_out);
  return static_cast<int32_t>(uidx.size());
}

// Slot schedule of fmt_sample_clips.  List scheduling in order of window count, descending (ties in input order): each clip goes to
// the slot that is free first (ties: the lowest slot) and starts at its own window 0 in the window that slot becomes free.
static const int kMaxSlots = 256;
static int list_schedule(const std::vector<int>& order, const int32_t* n_win, int n_slots, int32_t* slot, int32_t* start) {
  typedef std::pair<int, int> FreeAt;            // (first free window, slot)
  std::priority_queue<FreeAt, std::vector<FreeAt>, std::greater<FreeAt>> q;
  for (int k = 0; k < n_slots; ++k) q.push(FreeAt(0, k));
  int makespan = 0;
  for (int i : order) {
    const FreeAt f = q.top();
    q.pop();
    if (slot) slot[i] = f.second;
    if (start) start[i] = f.first;
    q.push(FreeAt(f.first + n_win[i], f.second));
    makespan = std::max(makespan, f.first + n_win[i]);
  }
  return makespan;
}

// n_slots = 0: the smallest slot count whose schedule ends with the longest clip (which bounds the call anyway), at most kMaxSlots
static int clip_schedule(int n, const int32_t* n_win, int n_slots, int32_t* slot, int32_t* start, int* makespan) {
  std::vector<int> order(n);
  long long total = 0;
  int longest = 0;
  for (int i = 0; i < n; ++i) { order[i] = i; total += n_win[i]; longest = std::max(longest, static_cast<int>(n_win[i])); }
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return n_win[a] > n_win[b]; });
  int S = n_slots;
  if (S == 0) {
    S = kMaxSlots;
    for (long long k = (total + longest - 1) / longest; k < kMaxSlots; ++k)      // fewer slots than total / longest cannot finish in time
      if (list_schedule(order, n_win, static_cast<int>(k), nullptr, nullptr) == longest) { S = static_cast<int>(k); break; }
  }
  *makespan = list_schedule(order, n_win, S, slot, start);
  return S;
}

int32_t fmt_occupancy_slots(int32_t plan_slots, int32_t n_ready) {
  if (plan_slots < 1 || plan_slots > kMaxSlots || n_ready < 1 || n_ready > plan_slots) return -1;
  int b = 1;
  while (b < n_ready) b *= 2;
  return b < plan_slots ? b : plan_slots;
}

int32_t fmt_clip_schedule(int32_t n_clips, const int32_t* n_windows, int32_t n_slots, int32_t* slot_out, int32_t* start_out, int32_t* makespan_out) {
  if (n_clips < 1 || n_windows == nullptr || n_slots < 0 || n_slots > kMaxSlots) return -1;
  for (int i = 0; i < n_clips; ++i)
    if (n_windows[i] < 1) return -1;
  int makespan = 0;
  const int S = clip_schedule(n_clips, n_windows, n_slots, slot_out, start_out, &makespan);
  if (makespan_out != nullptr) *makespan_out = makespan;
  return S;
}

// we_dynamic takes no part: no graph, table or buffer depends on it (each slot record carries its clip's emotion mode, and the
// condition-row map is the same for every mode, distinct_condition_rows), so a plan that differs only in it is the same plan.
// The occupancy buckets of a plan that runs one kernel per op: 1, 2, 4, ... slots below plan.batch, with the condition-row map of
// each (the plan's deduplication on its first B slots), uploaded here in one copy.  Their graphs are captured on first use.
static int make_buckets(FmtHandle* h, cudaStream_t st) {
  if (h->window_active) return 0;
  const ModelShape& s = h->shape;
  std::vector<int> maps;
  for (int B = 1; B < s.B; B *= 2) {
    FmtHandle::Bucket b;
    b.B = B;
    b.U = s.nb * B * s.N;
    if (h->dedup) {
      ModelShape sb = s;
      sb.B = B;
      std::vector<int> urow, uidx;
      const std::vector<int32_t> modes(B, h->plan.we_dynamic);
      distinct_condition_rows(sb, modes.data(), urow, uidx);
      b.U = static_cast<int>(uidx.size());
      b.map_off = maps.size();
      maps.insert(maps.end(), urow.begin(), urow.end());
      maps.insert(maps.end(), uidx.begin(), uidx.end());
    }
    h->buckets.push_back(b);
  }
  if (!maps.empty()) {
    FMT_OK(dev_alloc(h, h->bucket_maps, maps.size() * sizeof(int)));
    CUDA_OK(cudaMemcpyAsync(h->bucket_maps.p, maps.data(), maps.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaStreamSynchronize(st));          // `maps` is a stack object
  }
  return 0;
}

static bool same_plan(const FmtHandle* h, const FmtPlan* p) {
  if (!h->configured) return false;
  const FmtPlan& q = h->plan;
  if (q.batch != p->batch || q.n_branches != p->n_branches || q.mode != p->mode ||
      q.n_steps != p->n_steps || q.n_stages != p->n_stages)
    return false;
  const int ne = p->n_steps * p->n_stages;
  if (ne > 0 && memcmp(h->t_eval.data(), p->t_eval, ne * sizeof(float)) != 0) return false;
  if (p->n_steps > 0 && memcmp(h->dt.data(), p->dt, p->n_steps * sizeof(float)) != 0) return false;
  if (memcmp(h->rk_a.data(), p->rk_a, p->n_stages * p->n_stages * sizeof(float)) != 0) return false;
  if (memcmp(h->rk_b.data(), p->rk_b, p->n_stages * sizeof(float)) != 0) return false;
  return true;
}

int32_t fmt_configure(FmtHandle* h, const FmtPlan* p, void* stream) {
  REQUIRE(h && p, "fmt_configure: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_OK(cudaSetDevice(h->device));
  REQUIRE(p->batch >= 1, "fmt_configure: batch must be >= 1");
  REQUIRE(p->n_branches == 1 || p->n_branches == 3 || p->n_branches == 4, "fmt_configure: n_branches must be 1, 3 or 4");
  REQUIRE(p->mode == FMT_MODE_BF16 || p->mode == FMT_MODE_FP32_VALIDATE || p->mode == FMT_MODE_BF16X3, "fmt_configure: unknown mode %d", p->mode);
  REQUIRE(p->n_steps >= 0 && p->n_stages >= 1 && p->n_stages <= FMT_MAX_STAGES, "fmt_configure: bad n_steps/n_stages");
  REQUIRE(p->rk_a && p->rk_b && (p->n_steps == 0 || (p->t_eval && p->dt)), "fmt_configure: null schedule arrays");
  h->last_ode = false;
  if (same_plan(h, p)) {
    h->plan.we_dynamic = p->we_dynamic;    // the mode fmt_sample_clip, fmt_velocity and the calls without per-clip modes give every clip
    return 0;
  }
  if (p->mode == FMT_MODE_BF16X3) {
    FMT_OK(pack_split_all(h, st));
    CUDA_OK(cudaStreamSynchronize(st));
  }

  const FmtDims& d = h->d;
  const int ne = p->n_steps * p->n_stages;
  h->configured = false;
  if (h->graph_exec) { CUDA_OK(cudaStreamSynchronize(st)); cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; h->graph_nodes = 0; }
  if (h->ode_exec) { CUDA_OK(cudaStreamSynchronize(st)); cudaGraphExecDestroy(h->ode_exec); h->ode_exec = nullptr; }
  if (!h->buckets.empty()) { CUDA_OK(cudaStreamSynchronize(st)); drop_buckets(h); }
  h->ode_nodes = 0;
  h->s_chunk = 0;                                // the per-slot graph's condition rows are built again on first use
  h->plan = *p;
  h->t_eval.assign(p->t_eval, p->t_eval + ne);
  h->dt.assign(p->dt, p->dt + p->n_steps);
  h->rk_a.assign(p->rk_a, p->rk_a + p->n_stages * p->n_stages);
  h->rk_b.assign(p->rk_b, p->rk_b + p->n_stages);
  h->plan.t_eval = h->plan.dt = h->plan.rk_a = h->plan.rk_b = nullptr;
  h->n_eval = ne;

  ModelShape& s = h->shape;
  s.B = p->batch; s.nb = p->n_branches; s.N = h->N; s.P = d.num_prev_frames; s.L = d.frames_per_clip;
  s.W = d.dim_w; s.A = d.dim_a; s.E = d.dim_e; s.H = d.dim_h; s.Kc = h->Kc;
  branch_nulls(s);
  h->R = s.nb * s.B * s.N;
  h->U = h->R;
  // Distinct condition rows.  The CFG branches null whole inputs (FMT.py:360-392): the unconditional branch's current frames all see
  // [wr | 0 | 0] - ONE condition row per clip instead of L - and its context frames see [wr | prev_wa | 0], the same rows as the
  // audio-only branch's context frames (prev_wa is never nulled, prev_we is nulled like we).  c_embedder, SiLU and the AdaLN table
  // GEMM only depend on the condition row and the evaluation, so they run on the U distinct rows (121 of 180 per clip with 3-way
  // CFG) and every consumer of a table row goes through urow[].  Round 1's window kernels index the table by token row: plans that
  // could fall back to them keep U = R.
  h->dedup = false;
  {
    const bool old_window_plan = h->use_window != 0 && window_eligible(h, p) && !(h->use_window == 3 && flow_eligible(h, p));
    if (h->use_dedup && s.nb > 1 && !old_window_plan) {
      std::vector<int> urow, uidx;
      const std::vector<int32_t> modes(s.B, p->we_dynamic);
      distinct_condition_rows(s, modes.data(), urow, uidx);
      if (static_cast<int>(uidx.size()) < h->R) {
        h->U = static_cast<int>(uidx.size());
        h->dedup = true;
        FMT_OK(dev_alloc(h, h->urow_buf, urow.size() * sizeof(int)));
        FMT_OK(dev_alloc(h, h->uidx_buf, uidx.size() * sizeof(int)));
        CUDA_OK(cudaMemcpyAsync(h->urow_buf.p, urow.data(), urow.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        CUDA_OK(cudaMemcpyAsync(h->uidx_buf.p, uidx.data(), uidx.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        CUDA_OK(cudaStreamSynchronize(st));      // `urow` / `uidx` are stack objects
      }
    }
  }
  const size_t ts = p->mode == FMT_MODE_BF16 ? 2 : 4;   // bf16x3: 4-byte pairs, fp32 tables and QKV
  h->tsize = ts;
  const size_t R = h->R, U = h->U, H = s.H;
  // table chunking: the AdaLN tables of as many evaluations as fit in half of the memory that is free right now (what this handle
  // already holds for its tables counts as free: dev_alloc reuses it), at most 48 GB.  ComfyUI keeps the decoder and wav2vec models
  // on the same GPU, so a fixed cap could fail where the reference, with O(1 step) memory, succeeds; FMT_TABLE_GB overrides.
  const size_t per_eval = U * static_cast<size_t>(h->NT) * ts;
  size_t cap = static_cast<size_t>(48) << 30;
  {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
      const size_t avail = (free_b + h->table.bytes + h->silu.bytes) / 2;
      if (avail < cap) cap = avail;
    } else {
      (void)cudaGetLastError();
    }
    if (const char* e = getenv("FMT_TABLE_GB")) { const double gb = atof(e); if (gb > 0) cap = static_cast<size_t>(gb * (1u << 30)); }
  }
  size_t chunk = per_eval ? cap / per_eval : 1;
  if (chunk < 1) chunk = 1;
  if (chunk > static_cast<size_t>(ne > 0 ? ne : 1)) chunk = ne > 0 ? ne : 1;
  h->table_chunk = static_cast<int>(chunk);
  // the per-slot window graph (fmt_sample_clips_ode) keeps the truly-uncond current frames of a 4-branch plan one row per slot: B - 1
  // more condition rows, for which the table and SiLU buffers keep room, so that it always fits at least one evaluation
  const size_t slot_rows = h->dedup && s.nb == 4 ? static_cast<size_t>(s.B) - 1 : 0;

  const size_t nx = static_cast<size_t>(s.B) * s.L * s.W;
  FMT_OK(dev_alloc(h, h->cond, U * s.Kc * ts));
  FMT_OK(dev_alloc(h, h->cemb, U * H * 4));
  FMT_OK(dev_alloc(h, h->temb, static_cast<size_t>(ne > 0 ? ne : 1) * H * 4));
  FMT_OK(dev_alloc(h, h->tfreq, static_cast<size_t>(ne > 0 ? ne : 1) * 256 * 4));
  FMT_OK(dev_alloc(h, h->th, static_cast<size_t>(ne > 0 ? ne : 1) * H * 4));
  FMT_OK(dev_alloc(h, h->silu, (chunk * U + slot_rows) * H * ts));
  FMT_OK(dev_alloc(h, h->table, chunk * per_eval + slot_rows * h->NT * ts));
  FMT_OK(dev_alloc(h, h->xstate, nx * 4));
  FMT_OK(dev_alloc(h, h->ystage, nx * 4));
  FMT_OK(dev_alloc(h, h->kbuf, nx * 4 * p->n_stages));
  FMT_OK(dev_alloc(h, h->prevx, static_cast<size_t>(s.B) * (s.P > 0 ? s.P : 1) * s.W * 4));
  FMT_OK(dev_alloc(h, h->ax, R * s.W * ts));
  FMT_OK(dev_alloc(h, h->X, R * H * 4));
  FMT_OK(dev_alloc(h, h->A1, R * H * ts));
  FMT_OK(dev_alloc(h, h->QKV, R * 3 * H * ts));
  FMT_OK(dev_alloc(h, h->A2, R * H * ts));
  FMT_OK(dev_alloc(h, h->Hm, R * static_cast<size_t>(d.mlp_hidden) * ts));
  FMT_OK(dev_alloc(h, h->V, R * s.W * 4));
  FMT_OK(dev_alloc(h, h->ddt, static_cast<size_t>(p->n_steps > 0 ? p->n_steps : 1) * 4));
  FMT_OK(dev_alloc(h, h->dteval, static_cast<size_t>(ne > 0 ? ne : 1) * 4));
  FMT_OK(dev_alloc(h, h->wargs, sizeof(WindowArgs)));
  CUDA_OK(cudaMemsetAsync(h->prevx.p, 0, h->prevx.bytes, st));
  if (ne > 0) {
    // timestep embeddings of every evaluation (FMT.py:294), computed once per plan
    CUDA_OK(cudaMemcpyAsync(h->dteval.p, h->t_eval.data(), ne * sizeof(float), cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaMemcpyAsync(h->ddt.p, h->dt.data(), p->n_steps * sizeof(float), cudaMemcpyHostToDevice, st));
    timestep_freq_kernel<<<ne, 128, 0, st>>>(static_cast<const float*>(h->dteval.p), ne, static_cast<float*>(h->tfreq.p));
    LAUNCH_CHECK(); count_launch(h);
    const int w1 = ne * s.H;
    small_linear_kernel<<<(w1 * 32 + 255) / 256, 256, 0, st>>>(static_cast<const float*>(h->tfreq.p), h->t0_w, h->t0_b, static_cast<float*>(h->th.p), ne, s.H, 256, 1);
    LAUNCH_CHECK(); count_launch(h);
    small_linear_kernel<<<(w1 * 32 + 255) / 256, 256, 0, st>>>(static_cast<const float*>(h->th.p), h->t2_w, h->t2_b, static_cast<float*>(h->temb.p), ne, s.H, s.H, 0);
    LAUNCH_CHECK(); count_launch(h);
    CUDA_OK(cudaStreamSynchronize(st));   // t_eval/dt host vectors may be reassigned by the next configure
  }

  // dataflow kernel first (FMT_WINDOW=3, the default); its setup fails soft: the plan then runs one kernel per op
  h->flow_active = false;
  if (flow_eligible(h, p) && h->table_chunk == ne) {
    if (setup_flow(h, st) == 0 && launch_flow(h, st, /*probe_only=*/true) == 0) h->flow_active = true;
    else (void)cudaGetLastError();
  }
  h->window_active = h->flow_active || (window_eligible(h, p) && h->table_chunk == ne && !h->dedup);   // round 1's kernels index the table by token row
  if (h->window_active && !h->flow_active) {
    // the persistent kernel synchronises across the grid: it needs one resident CTA on every SM, else the plan runs one kernel per op
    int occ = 0;
    cudaError_t oe = cudaErrorUnknown;
    switch (d.dim_h / 128) {
      case 1: oe = cudaFuncSetAttribute(fmt_window_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, WIN_SMEM_BYTES);
              if (oe == cudaSuccess) oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fmt_window_kernel<1, false>, WIN_THREADS, WIN_SMEM_BYTES); break;
      case 2: oe = cudaFuncSetAttribute(fmt_window_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, WIN_SMEM_BYTES);
              if (oe == cudaSuccess) oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fmt_window_kernel<2, false>, WIN_THREADS, WIN_SMEM_BYTES); break;
      case 4: oe = cudaFuncSetAttribute(fmt_window_kernel<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, WIN_SMEM_BYTES);
              if (oe == cudaSuccess) oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fmt_window_kernel<4, false>, WIN_THREADS, WIN_SMEM_BYTES); break;
      case 8: oe = cudaFuncSetAttribute(fmt_window_kernel<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, WIN_SMEM_BYTES);
              if (oe == cudaSuccess) oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fmt_window_kernel<8, false>, WIN_THREADS, WIN_SMEM_BYTES); break;
    }
    if (oe != cudaSuccess || occ < 1) { (void)cudaGetLastError(); h->window_active = false; }
  }
  if (h->window_active && !h->flow_active) FMT_OK(setup_window(h, st));

  // capture one window as a CUDA graph
  h->ksliced = false;
  FMT_OK(capture_window(h, enqueue_window_mode, plan_graph(h), &h->graph_exec, &h->graph_nodes, &h->capture_launches));
  h->plan_ksliced = h->ksliced;
  FMT_OK(make_buckets(h, st));
  h->configured = true;
  return 0;
}

static int set_wargs(FmtHandle* h, const WindowArgs& a, cudaStream_t st) {
  set_window_args_kernel<<<1, 1, 0, st>>>(static_cast<WindowArgs*>(h->wargs.p), a);
  LAUNCH_CHECK(); count_launch(h);
  return 0;
}

// Slot records of one call (every sampling entry point and fmt_velocity) go up in ONE copy from a pinned staging buffer that the handle
// owns; slot_ev marks the end of the previous call's copy, so the staging buffer is refilled only once that copy has read it.
// stage_slot_records fills the staging buffer with n_win windows of `slots` idle records each (the slots of the window graph the call
// replays): zero inputs ((L, W) noise, and r_s / wa / we rows no wider than that), no output, no context, static emotion, scales of 1
// and the plan's branch count; with ode, `slots` SlotOde follow the SlotArgs of each window, idle as well (no evaluation).
static int stage_slot_records(FmtHandle* h, size_t n_win, bool ode, int slots, cudaStream_t st) {
  const ModelShape& s = h->shape;
  if (!h->slot_zero.p) {   // its size depends on the model's dims alone, and no kernel writes it: zeroed once per handle
    const size_t n_zero = std::max<size_t>(static_cast<size_t>(s.L) * s.W, static_cast<size_t>(std::max(s.A, s.E)));
    FMT_OK(dev_alloc(h, h->slot_zero, n_zero * sizeof(float)));
    CUDA_OK(cudaMemsetAsync(h->slot_zero.p, 0, n_zero * sizeof(float), st));
  }
  const float* zero = static_cast<const float*>(h->slot_zero.p);
  if (h->slot_ev) CUDA_OK(cudaEventSynchronize(h->slot_ev));
  h->slot_recs = slots;
  h->slot_stride = static_cast<size_t>(slots) * (sizeof(SlotArgs) + (ode ? sizeof(SlotOde) : 0));
  const size_t bytes = n_win * h->slot_stride;
  if (h->slot_host_bytes < bytes) {
    if (h->slot_host) { CUDA_OK(cudaFreeHost(h->slot_host)); h->slot_host = nullptr; h->slot_host_bytes = 0; }
    CUDA_OK(cudaHostAlloc(reinterpret_cast<void**>(&h->slot_host), bytes, cudaHostAllocDefault));
    h->slot_host_bytes = bytes;
  }
  for (size_t w = 0; w < n_win; ++w) {
    SlotArgs* rec = reinterpret_cast<SlotArgs*>(h->slot_host + w * h->slot_stride);
    for (int k = 0; k < slots; ++k) {
      SlotArgs& z = rec[k];
      z.r_s = zero; z.wa = zero; z.we = zero; z.x0 = zero; z.r_d = nullptr; z.ctx = nullptr;
      z.T_wa = 1; z.T_we = 1; z.T_out = 0; z.win_start = 0; z.out_start = 0; z.first_window = 1;
      z.a_scale = z.r_scale = z.e_scale = 1.f; z.n_branches = s.nb; z.we_dynamic = 0;
    }
    if (!ode) continue;
    SlotOde* od = reinterpret_cast<SlotOde*>(rec + slots);
    for (int k = 0; k < slots; ++k) {
      SlotOde& o = od[k];
      o = SlotOde{};
      o.temb = static_cast<const float*>(h->temb.p); o.dt = static_cast<const float*>(h->ddt.p); o.n_eval = 0; o.n_stages = 1;
    }
  }
  return 0;
}

// window w's SlotArgs / SlotOde in the staging buffer, and its SlotArgs on the device after upload_slot_records
static SlotArgs* staged_args(FmtHandle* h, size_t w) { return reinterpret_cast<SlotArgs*>(h->slot_host + w * h->slot_stride); }
static SlotOde* staged_ode(FmtHandle* h, size_t w) { return reinterpret_cast<SlotOde*>(staged_args(h, w) + h->slot_recs); }
static const SlotArgs* device_args(const FmtHandle* h, size_t w) {
  return reinterpret_cast<const SlotArgs*>(static_cast<const unsigned char*>(h->slot_buf.p) + w * h->slot_stride);
}

static int upload_slot_records(FmtHandle* h, size_t n_win, cudaStream_t st) {
  const size_t bytes = n_win * h->slot_stride;
  FMT_OK(dev_alloc(h, h->slot_buf, bytes));
  CUDA_OK(cudaMemcpyAsync(h->slot_buf.p, h->slot_host, bytes, cudaMemcpyHostToDevice, st));
  if (!h->slot_ev) CUDA_OK(cudaEventCreateWithFlags(&h->slot_ev, cudaEventDisableTiming));
  CUDA_OK(cudaEventRecord(h->slot_ev, st));
  return 0;
}

// ---- per-slot ODE schedules
// Checks the schedule of every one of n clips / streams against the plan: at most the plan's evaluations, 1..FMT_MAX_STAGES stages.
static int check_odes(const FmtHandle* h, const FmtClipOde* ode, int n, const char* who) {
  REQUIRE(ode->n_steps && ode->n_stages && ode->t_eval && ode->dt && ode->rk_a && ode->rk_b, "%s: null ODE array", who);
  for (int i = 0; i < n; ++i) {
    const int S = ode->n_steps[i], G = ode->n_stages[i];
    REQUIRE(G >= 1 && G <= FMT_MAX_STAGES && S >= 0, "%s: %d: n_steps=%d, n_stages=%d (1..%d)", who, i, S, G, FMT_MAX_STAGES);
    REQUIRE(static_cast<long long>(S) * G <= h->n_eval, "%s: %d needs %lld evaluations per window, the plan runs %d", who, i,
            static_cast<long long>(S) * G, h->n_eval);
    REQUIRE(ode->rk_a[i] && ode->rk_b[i] && (S == 0 || (ode->t_eval[i] && ode->dt[i])), "%s: %d: null schedule array", who, i);
  }
  return 0;
}

// Slot record of schedule i, with its t-embeddings and step sizes on the device: the plan's own when the schedule is the plan's,
// else computed once per distinct schedule (timestep_freq_kernel and the two small_linear_kernel launches of fmt_configure, so the
// same t gives the same bits) and kept in the handle.  A schedule without evaluations points at the plan's.
static int slot_ode(FmtHandle* h, const FmtClipOde* ode, int i, cudaStream_t st, SlotOde* out) {
  const int S = ode->n_steps[i], G = ode->n_stages[i], ne = S * G, H = h->shape.H;
  SlotOde o{};
  o.n_eval = ne; o.n_stages = G;
  for (int g = 0; g < G; ++g) {
    for (int j = 0; j < G; ++j) o.rk_a[g * 4 + j] = ode->rk_a[i][g * G + j];
    o.rk_b[g] = ode->rk_b[i][g];
  }
  o.temb = static_cast<const float*>(h->temb.p); o.dt = static_cast<const float*>(h->ddt.p);
  const bool plan = S == h->plan.n_steps && G == h->plan.n_stages && (ne == 0 || (memcmp(ode->t_eval[i], h->t_eval.data(), ne * sizeof(float)) == 0 &&
                    memcmp(ode->dt[i], h->dt.data(), S * sizeof(float)) == 0));
  if (ne > 0 && !plan) {
    std::vector<float> key(ode->t_eval[i], ode->t_eval[i] + ne);
    key.insert(key.end(), ode->dt[i], ode->dt[i] + S);
    key.push_back(static_cast<float>(S));
    auto it = h->ode_cache.find(key);
    if (it == h->ode_cache.end()) {
      DevBuf buf;
      FMT_OK(dev_alloc(h, buf, (static_cast<size_t>(ne) * H + S) * sizeof(float)));
      it = h->ode_cache.emplace(key, buf).first;
      float* temb = static_cast<float*>(buf.p);
      // dteval / tfreq / th hold the plan's evaluations (>= ne) and are only read while t-embeddings are computed
      CUDA_OK(cudaMemcpyAsync(h->dteval.p, ode->t_eval[i], ne * sizeof(float), cudaMemcpyHostToDevice, st));
      CUDA_OK(cudaMemcpyAsync(temb + static_cast<size_t>(ne) * H, ode->dt[i], S * sizeof(float), cudaMemcpyHostToDevice, st));
      timestep_freq_kernel<<<ne, 128, 0, st>>>(static_cast<const float*>(h->dteval.p), ne, static_cast<float*>(h->tfreq.p));
      LAUNCH_CHECK(); count_launch(h);
      const int w1 = ne * H;
      small_linear_kernel<<<(w1 * 32 + 255) / 256, 256, 0, st>>>(static_cast<const float*>(h->tfreq.p), h->t0_w, h->t0_b, static_cast<float*>(h->th.p), ne, H, 256, 1);
      LAUNCH_CHECK(); count_launch(h);
      small_linear_kernel<<<(w1 * 32 + 255) / 256, 256, 0, st>>>(static_cast<const float*>(h->th.p), h->t2_w, h->t2_b, temb, ne, H, H, 0);
      LAUNCH_CHECK(); count_launch(h);
      CUDA_OK(cudaStreamSynchronize(st));   // the caller's host arrays may go away after the call
    }
    o.temb = static_cast<const float*>(it->second.p);
    o.dt = o.temb + static_cast<size_t>(ne) * H;
  }
  *out = o;
  return 0;
}

// The per-slot window graph of the current plan, captured on first use: its distinct condition rows (the plan's deduplication with
// no row shared between slots), their buffers, and a kbuf of FMT_MAX_STAGES stages.  The AdaLN tables go to the plan's table buffer,
// as many evaluations at a time as it holds.
static int ensure_ode_rows(FmtHandle* h, cudaStream_t st) {
  if (h->s_chunk > 0) return 0;
  const ModelShape& s = h->shape;
  h->sU = h->R;
  h->s_dedup = false;
  if (h->use_dedup && s.nb > 1) {
    std::vector<int> urow, uidx;
    const std::vector<int32_t> modes(s.B, h->plan.we_dynamic);
    distinct_condition_rows(s, modes.data(), urow, uidx, true);
    if (static_cast<int>(uidx.size()) < h->R) {
      h->sU = static_cast<int>(uidx.size());
      h->s_dedup = true;
      FMT_OK(dev_alloc(h, h->s_urow, urow.size() * sizeof(int)));
      FMT_OK(dev_alloc(h, h->s_uidx, uidx.size() * sizeof(int)));
      CUDA_OK(cudaMemcpyAsync(h->s_urow.p, urow.data(), urow.size() * sizeof(int), cudaMemcpyHostToDevice, st));
      CUDA_OK(cudaMemcpyAsync(h->s_uidx.p, uidx.data(), uidx.size() * sizeof(int), cudaMemcpyHostToDevice, st));
      CUDA_OK(cudaStreamSynchronize(st));      // `urow` / `uidx` are stack objects
    }
  }
  const size_t U = h->sU, ts = h->tsize, nx = static_cast<size_t>(s.B) * s.L * s.W;
  const size_t by_table = h->table.bytes / (U * h->NT * ts), by_silu = h->silu.bytes / (U * s.H * ts);
  const size_t chunk = h->n_eval == 0 ? 1 : std::min<size_t>(std::min(by_table, by_silu), h->n_eval);
  REQUIRE(chunk >= 1, "per-slot schedules: the AdaLN table buffer holds no evaluation of %zu condition rows", U);   // fmt_configure keeps room
  h->s_chunk = static_cast<int>(chunk);
  FMT_OK(dev_alloc(h, h->s_cond, U * s.Kc * ts));
  FMT_OK(dev_alloc(h, h->s_cemb, U * s.H * 4));
  FMT_OK(dev_alloc(h, h->s_kbuf, nx * 4 * FMT_MAX_STAGES));
  return 0;
}

static int ensure_ode_graph(FmtHandle* h, cudaStream_t st) {
  if (h->ode_exec) return 0;
  FMT_OK(ensure_ode_rows(h, st));
  return capture_window(h, enqueue_window_ode_mode, plan_graph(h, true), &h->ode_exec, &h->ode_nodes, &h->ode_launches);
}

// ---- occupancy buckets
// A bucket's graphs: the plan's GraphShape on its first B slots, with the bucket's condition-row map in the plan's buffers
static GraphShape bucket_graph(const FmtHandle* h, const FmtHandle::Bucket& b, bool ode) {
  GraphShape g = plan_graph(h, ode);
  g.s.B = b.B;
  g.R = g.s.nb * b.B * g.s.N;
  g.ksplit = h->plan_ksliced;
  CondRows& r = g.rows;
  r.U = ode ? b.sU : b.U;
  const int* map = ode ? (h->s_dedup ? static_cast<const int*>(b.s_map.p) : nullptr)
                       : (h->dedup ? static_cast<const int*>(h->bucket_maps.p) + b.map_off : nullptr);
  r.urow = map;
  r.uidx = map ? map + g.R : nullptr;
  return g;
}

// Bucket b's window graph (ode: its per-slot window graph), captured the first time a step needs it.  It holds the kernels of the
// plan's graph of the same kind, one for one.
static int ensure_bucket_graph(FmtHandle* h, FmtHandle::Bucket& b, bool ode, cudaStream_t st) {
  if (ode ? b.ode_exec != nullptr : b.exec != nullptr) return 0;
  if (ode) {
    FMT_OK(ensure_ode_rows(h, st));
    const ModelShape& s = h->shape;
    b.sU = s.nb * b.B * s.N;
    if (h->s_dedup) {   // the plan's per-slot graph shares no row between slots, so neither does the bucket's
      ModelShape sb = s;
      sb.B = b.B;
      std::vector<int> urow, uidx;
      const std::vector<int32_t> modes(b.B, h->plan.we_dynamic);
      distinct_condition_rows(sb, modes.data(), urow, uidx, true);
      b.sU = static_cast<int>(uidx.size());
      urow.insert(urow.end(), uidx.begin(), uidx.end());
      FMT_OK(dev_alloc(h, b.s_map, urow.size() * sizeof(int)));
      CUDA_OK(cudaMemcpyAsync(b.s_map.p, urow.data(), urow.size() * sizeof(int), cudaMemcpyHostToDevice, st));
      CUDA_OK(cudaStreamSynchronize(st));      // `urow` is a stack object
    }
  }
  cudaGraphExec_t exec = nullptr;
  int nodes = 0;
  long long launches = 0;
  FMT_OK(capture_window(h, ode ? enqueue_window_ode_mode : enqueue_window_mode, bucket_graph(h, b, ode), &exec, &nodes, &launches));
  if (ode && h->ode_nodes == 0) h->ode_nodes = nodes;   // every bucket's per-slot graph has the same kernels
  if (nodes != (ode ? h->ode_nodes : h->graph_nodes)) {
    cudaGraphExecDestroy(exec);
    return set_err(-2, "occupancy bucket of %d slots: its graph has %d nodes, the plan's %d", b.B, nodes, ode ? h->ode_nodes : h->graph_nodes);
  }
  (ode ? b.ode_exec : b.exec) = exec;
  (ode ? b.ode_launches : b.launches) = launches;
  return 0;
}

// One clip as its slot records see it: tensors of that clip alone (batch 1), the noise of its window w at noise + w * noise_stride,
// and its guidance
struct ClipIn {
  const float *r_s, *wa, *we, *noise;
  float* r_d;
  size_t noise_stride;
  int T_wa, T_we, T;
  float a_scale, r_scale, e_scale;
  int n_branches;
  int we_dynamic;
};

// The rules every clip of fmt_sample_clip / fmt_sample_clips follows, those of its own emotion mode among them; `who` names it in the
// error.  *n_win: its window count.
static int check_clip(const ModelShape& s, const ClipIn& c, const char* who, int32_t* n_win) {
  const int nb = c.n_branches;
  REQUIRE((nb == 1 || nb == 3 || nb == 4) && nb <= s.nb, "%s: n_branches=%d must be 1, 3 or 4 and fit the plan's %d branches", who, nb, s.nb);
  REQUIRE(c.r_s && c.wa && c.we && c.noise && c.r_d, "%s: null tensor pointer", who);
  REQUIRE(c.T >= 1 && c.T_wa >= 1 && c.T_we >= 1, "%s: empty clip", who);
  REQUIRE(c.we_dynamic == 0 || c.we_dynamic == 1, "%s: we_dynamic=%d must be 0 or 1", who, c.we_dynamic);
  REQUIRE(c.we_dynamic ? c.T_we > 1 : c.T_we == 1, "%s: T_we=%d does not match we_dynamic=%d", who, c.T_we, c.we_dynamic);
  const int n = (c.T + s.L - 1) / s.L;
  // every window must see at least one real wa (and dynamic we) frame; the reference's F.pad(replicate) fails otherwise
  REQUIRE((n - 1) * s.L < c.T_wa, "%s: wa has %d frames but window %d starts at frame %d", who, c.T_wa, n - 1, (n - 1) * s.L);
  REQUIRE(!c.we_dynamic || (n - 1) * s.L < c.T_we, "%s: dynamic we has %d frames but the last window starts at %d", who, c.T_we, (n - 1) * s.L);
  *n_win = n;
  return 0;
}

// Stages the slot records of `makespan` windows in which clip i runs its window w in slot slot[i] of window start[i] + w, every
// other slot idle; od: the clips' SlotOde for the per-slot window graph (empty: the plan's graph).
static int stage_clips(FmtHandle* h, const std::vector<ClipIn>& c, const int32_t* slot, const int32_t* start, int makespan,
                       const std::vector<SlotOde>& od, cudaStream_t st) {
  const ModelShape& s = h->shape;
  FMT_OK(stage_slot_records(h, makespan, !od.empty(), s.B, st));
  for (size_t i = 0; i < c.size(); ++i) {
    const int n_win = (c[i].T + s.L - 1) / s.L;
    for (int w = 0; w < n_win; ++w) {
      if (!od.empty()) staged_ode(h, start[i] + w)[slot[i]] = od[i];
      SlotArgs& z = staged_args(h, start[i] + w)[slot[i]];
      z.r_s = c[i].r_s; z.wa = c[i].wa; z.we = c[i].we; z.r_d = c[i].r_d;
      z.x0 = c[i].noise + w * c[i].noise_stride;
      z.T_wa = c[i].T_wa; z.T_we = c[i].T_we; z.T_out = c[i].T;
      z.win_start = z.out_start = w * s.L; z.first_window = (w == 0);
      z.a_scale = c[i].a_scale; z.r_scale = c[i].r_scale; z.e_scale = c[i].e_scale; z.n_branches = c[i].n_branches;
      z.we_dynamic = c[i].we_dynamic;
    }
  }
  return 0;
}

// Uploads the staged records of n_win windows and replays a window graph once per window: the plan's, or with ode the per-slot one
// (bk: those of an occupancy bucket)
static int replay_windows(FmtHandle* h, int n_win, bool ode, fmt_progress_fn progress, void* progress_user, cudaStream_t st,
                          const FmtHandle::Bucket* bk = nullptr) {
  cudaGraphExec_t exec = bk ? (ode ? bk->ode_exec : bk->exec) : (ode ? h->ode_exec : h->graph_exec);
  const long long n_launch = bk ? (ode ? bk->ode_launches : bk->launches) : (ode ? h->ode_launches : h->capture_launches);
  FMT_OK(upload_slot_records(h, n_win, st));
  h->last_ode = ode;
  h->last_slots = bk ? bk->B : h->shape.B;
  for (int w = 0; w < n_win; ++w) {
    FMT_OK(set_wargs(h, WindowArgs{device_args(h, w)}, st));
    CUDA_OK(cudaGraphLaunch(exec, st));
    h->launches += n_launch;
    if (progress) progress(w, n_win, progress_user);
  }
  return 0;
}

int32_t fmt_sample_clip(FmtHandle* h, const FmtClip* c, void* stream) {
  REQUIRE(h && c, "fmt_sample_clip: null argument");
  REQUIRE(h->configured, "fmt_sample_clip: call fmt_configure first");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_OK(cudaSetDevice(h->device));
  const ModelShape& s = h->shape;
  ClipIn in{c->r_s, c->wa, c->we, c->noise, c->r_d, 0, c->T_wa, c->T_we, c->audio_num_frames, c->a_cfg_scale, c->r_cfg_scale, c->e_cfg_scale, s.nb,
             h->plan.we_dynamic};
  int32_t n_win = 0;
  FMT_OK(check_clip(s, in, "fmt_sample_clip", &n_win));
  const int T = in.T;
  const size_t n_rs = static_cast<size_t>(s.B) * s.W, n_wa = static_cast<size_t>(s.B) * in.T_wa * s.A, n_we = static_cast<size_t>(s.B) * in.T_we * s.E;
  const size_t n_noise = static_cast<size_t>(n_win) * s.B * s.L * s.W, n_rd = static_cast<size_t>(s.B) * T * s.W;
  if (c->location == FMT_LOC_HOST) {
    FMT_OK(dev_alloc(h, h->st_rs, n_rs * 4)); FMT_OK(dev_alloc(h, h->st_wa, n_wa * 4)); FMT_OK(dev_alloc(h, h->st_we, n_we * 4));
    FMT_OK(dev_alloc(h, h->st_noise, n_noise * 4)); FMT_OK(dev_alloc(h, h->st_rd, n_rd * 4));
    CUDA_OK(cudaMemcpyAsync(h->st_rs.p, in.r_s, n_rs * 4, cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaMemcpyAsync(h->st_wa.p, in.wa, n_wa * 4, cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaMemcpyAsync(h->st_we.p, in.we, n_we * 4, cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaMemcpyAsync(h->st_noise.p, in.noise, n_noise * 4, cudaMemcpyHostToDevice, st));
    in.r_s = static_cast<float*>(h->st_rs.p); in.wa = static_cast<float*>(h->st_wa.p); in.we = static_cast<float*>(h->st_we.p);
    in.noise = static_cast<float*>(h->st_noise.p); in.r_d = static_cast<float*>(h->st_rd.p);
  }
  // batch row b is slot b of every window: its rows of the batched tensors, the noise of its window w at noise[w][b]
  std::vector<ClipIn> rows(s.B, in);
  std::vector<int32_t> slot(s.B), start(s.B, 0);
  for (int b = 0; b < s.B; ++b) {
    ClipIn& r = rows[b];
    r.r_s += static_cast<size_t>(b) * s.W;
    r.wa += static_cast<size_t>(b) * in.T_wa * s.A;
    r.we += static_cast<size_t>(b) * in.T_we * s.E;
    r.noise += static_cast<size_t>(b) * s.L * s.W;
    r.noise_stride = static_cast<size_t>(s.B) * s.L * s.W;
    r.r_d += static_cast<size_t>(b) * T * s.W;
    slot[b] = b;
  }
  FMT_OK(stage_clips(h, rows, slot.data(), start.data(), n_win, {}, st));
  FMT_OK(replay_windows(h, n_win, false, c->progress, c->progress_user, st));
  if (c->location == FMT_LOC_HOST) {
    CUDA_OK(cudaMemcpyAsync(c->r_d, in.r_d, n_rd * 4, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    // the persistent kernels report a tripped bounded spin through a mapped status word (the launch fails as well)
    if (h->window_active && h->win_err_host && *h->win_err_host != 0) return set_err(-6, "window kernel reported status 0x%08x", *h->win_err_host);
  }
  return 0;
}

// Many clips on plan.batch slots: window w of the call runs, in slot k, whichever clip the schedule put there (at that clip's own
// window), through the same captured window graph (ode != nullptr: each clip on its own schedule, through the per-slot window graph).
// g == nullptr: the set's scales and the plan's branch count for every clip; we_dyn == nullptr: plan.we_dynamic for every clip.
int32_t fmt_sample_clip_set(FmtHandle* h, const FmtClipSet* cs, const FmtClipGuidance* g, const FmtClipOde* ode, const int32_t* we_dyn,
                            void* stream) {
  REQUIRE(h && cs, "fmt_sample_clips: null argument");
  REQUIRE(h->configured, "fmt_sample_clips: call fmt_configure first");
  const int n = cs->n_clips;
  REQUIRE(n >= 1, "fmt_sample_clips: no clips");
  REQUIRE(cs->r_s && cs->wa && cs->we && cs->noise && cs->r_d && cs->T_wa && cs->T_we && cs->audio_num_frames, "fmt_sample_clips: null array");
  REQUIRE(!g || (g->a_cfg_scale && g->r_cfg_scale && g->e_cfg_scale && g->n_branches), "fmt_sample_clips_guided: null guidance array");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_OK(cudaSetDevice(h->device));
  const ModelShape& s = h->shape;
  std::vector<ClipIn> c(n);
  std::vector<int32_t> n_win(n), slot(n), start(n);
  for (int i = 0; i < n; ++i) {
    c[i] = ClipIn{cs->r_s[i], cs->wa[i], cs->we[i], cs->noise[i], cs->r_d[i], static_cast<size_t>(s.L) * s.W, cs->T_wa[i], cs->T_we[i],
                  cs->audio_num_frames[i], g ? g->a_cfg_scale[i] : cs->a_cfg_scale, g ? g->r_cfg_scale[i] : cs->r_cfg_scale,
                  g ? g->e_cfg_scale[i] : cs->e_cfg_scale, g ? g->n_branches[i] : s.nb, we_dyn ? we_dyn[i] : h->plan.we_dynamic};
    char who[48];
    snprintf(who, sizeof(who), "fmt_sample_clips: clip %d", i);
    FMT_OK(check_clip(s, c[i], who, &n_win[i]));
  }
  if (ode) FMT_OK(check_odes(h, ode, n, "fmt_sample_clips_ode: clip"));
  int makespan = 0;
  const int S = clip_schedule(n, n_win.data(), 0, slot.data(), start.data(), &makespan);
  REQUIRE(s.B == S, "fmt_sample_clips: the plan has batch %d, but these %d clips are scheduled on %d slots (fmt_clip_schedule)", s.B, n, S);

  std::vector<SlotOde> od(ode ? n : 0);
  for (int i = 0; i < static_cast<int>(od.size()); ++i) FMT_OK(slot_ode(h, ode, i, st, &od[i]));
  if (ode) FMT_OK(ensure_ode_graph(h, st));
  FMT_OK(stage_clips(h, c, slot.data(), start.data(), makespan, od, st));
  return replay_windows(h, makespan, ode != nullptr, cs->progress, cs->progress_user, st);
}

int32_t fmt_sample_clips(FmtHandle* h, const FmtClipSet* cs, void* stream) { return fmt_sample_clip_set(h, cs, nullptr, nullptr, nullptr, stream); }

int32_t fmt_sample_clips_guided(FmtHandle* h, const FmtClipSet* cs, const FmtClipGuidance* g, void* stream) {
  REQUIRE(g, "fmt_sample_clips_guided: null argument");
  return fmt_sample_clip_set(h, cs, g, nullptr, nullptr, stream);
}

int32_t fmt_sample_clips_ode(FmtHandle* h, const FmtClipSet* cs, const FmtClipGuidance* g, const FmtClipOde* ode, void* stream) {
  REQUIRE(g, "fmt_sample_clips_guided: null argument");
  return fmt_sample_clip_set(h, cs, g, ode, nullptr, stream);
}

// One window of each of n streams, stream i in slot i, through the captured window graph of fmt_occupancy_slots(batch, n) slots (ode !=
// nullptr: each stream on its own schedule, through the per-slot window graph of those slots); its slots n.. are idle.  A plan whose
// window graph is a persistent kernel replays its one graph of batch slots.  A stream's context lives in its own ctx buffer, not in the
// handle, so a stream may run in any slot and the plan may be replaced between calls.  Its wa / we start at the window's first
// context frame (P frames before its first current frame), or at its first current frame in a first window; its output is the
// window alone.  we_dyn == nullptr: plan.we_dynamic for every stream.
int32_t fmt_sample_window_set(FmtHandle* h, const FmtWindowSet* ws, const FmtClipGuidance* g, const FmtClipOde* ode, const int32_t* we_dyn,
                              void* stream) {
  REQUIRE(h && ws && g, "fmt_sample_windows: null argument");
  REQUIRE(h->configured, "fmt_sample_windows: call fmt_configure first");
  const ModelShape& s = h->shape;
  const int n = ws->n_streams;
  REQUIRE(n >= 1 && n <= s.B, "fmt_sample_windows: %d streams, the plan has %d slots", n, s.B);
  REQUIRE(ws->r_s && ws->wa && ws->we && ws->x0 && ws->ctx && ws->r_d && ws->T_wa && ws->T_we && ws->n_out && ws->first_window,
          "fmt_sample_windows: null array");
  REQUIRE(g->a_cfg_scale && g->r_cfg_scale && g->e_cfg_scale && g->n_branches, "fmt_sample_windows: null guidance array");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_OK(cudaSetDevice(h->device));
  for (int i = 0; i < n; ++i) {
    const int nb = g->n_branches[i];
    REQUIRE((nb == 1 || nb == 3 || nb == 4) && nb <= s.nb,
            "fmt_sample_windows: stream %d: n_branches=%d must be 1, 3 or 4 and fit the plan's %d branches", i, nb, s.nb);
    REQUIRE(ws->r_s[i] && ws->wa[i] && ws->we[i] && ws->x0[i] && ws->ctx[i] && ws->r_d[i], "fmt_sample_windows: stream %d: null tensor pointer", i);
    const int first = ws->first_window[i], T_wa = ws->T_wa[i], T_we = ws->T_we[i], n_out = ws->n_out[i];
    const int dyn = we_dyn ? we_dyn[i] : h->plan.we_dynamic;
    REQUIRE(first == 0 || first == 1, "fmt_sample_windows: stream %d: first_window=%d must be 0 or 1", i, first);
    REQUIRE(n_out >= 1 && n_out <= s.L, "fmt_sample_windows: stream %d: n_out=%d outside [1, %d]", i, n_out, s.L);
    REQUIRE(dyn == 0 || dyn == 1, "fmt_sample_windows: stream %d: we_dynamic=%d must be 0 or 1", i, dyn);
    REQUIRE(dyn ? T_we >= 1 : T_we == 1, "fmt_sample_windows: stream %d: T_we=%d does not match we_dynamic=%d", i, T_we, dyn);
    // the window's first current frame must be a real frame (the reference's F.pad(replicate) fails otherwise)
    const int cur = first ? 0 : s.P;
    REQUIRE(cur < T_wa, "fmt_sample_windows: stream %d: wa has %d frames but the window's first current frame is frame %d", i, T_wa, cur);
    REQUIRE(!dyn || cur < T_we, "fmt_sample_windows: stream %d: dynamic we has %d frames but the window's first current frame is frame %d",
            i, T_we, cur);
  }
  if (ode) FMT_OK(check_odes(h, ode, n, "fmt_sample_windows_ode: stream"));
  std::vector<SlotOde> od(ode ? n : 0);
  for (int i = 0; i < static_cast<int>(od.size()); ++i) FMT_OK(slot_ode(h, ode, i, st, &od[i]));
  // the graphs of the occupancy bucket of n streams; a plan whose window graph is a persistent kernel has no buckets
  const int slots = h->buckets.empty() ? s.B : fmt_occupancy_slots(s.B, n);
  FmtHandle::Bucket* bk = nullptr;
  if (slots < s.B) {
    bk = &h->buckets[__builtin_ctz(static_cast<unsigned>(slots))];   // bucket i holds 2^i slots
    FMT_OK(ensure_bucket_graph(h, *bk, ode != nullptr, st));
  } else if (ode) {
    FMT_OK(ensure_ode_graph(h, st));
  }
  FMT_OK(stage_slot_records(h, 1, ode != nullptr, slots, st));
  for (int i = 0; i < n; ++i) {
    if (ode) staged_ode(h, 0)[i] = od[i];
    SlotArgs& z = staged_args(h, 0)[i];
    z.r_s = ws->r_s[i]; z.wa = ws->wa[i]; z.we = ws->we[i]; z.x0 = ws->x0[i]; z.r_d = ws->r_d[i]; z.ctx = ws->ctx[i];
    z.T_wa = ws->T_wa[i]; z.T_we = ws->T_we[i]; z.T_out = ws->n_out[i];
    z.first_window = ws->first_window[i];
    z.win_start = z.first_window ? 0 : s.P; z.out_start = 0;
    z.a_scale = g->a_cfg_scale[i]; z.r_scale = g->r_cfg_scale[i]; z.e_scale = g->e_cfg_scale[i]; z.n_branches = g->n_branches[i];
    z.we_dynamic = we_dyn ? we_dyn[i] : h->plan.we_dynamic;
  }
  return replay_windows(h, 1, ode != nullptr, nullptr, nullptr, st, bk);
}

int32_t fmt_sample_windows(FmtHandle* h, const FmtWindowSet* ws, const FmtClipGuidance* g, void* stream) {
  return fmt_sample_window_set(h, ws, g, nullptr, nullptr, stream);
}

int32_t fmt_sample_windows_ode(FmtHandle* h, const FmtWindowSet* ws, const FmtClipGuidance* g, const FmtClipOde* ode, void* stream) {
  return fmt_sample_window_set(h, ws, g, ode, nullptr, stream);
}

}  // extern "C"

// dst (B, P + L, C) <- [prev (B, P, C) | cur (B, L, C)] of every clip (device pointers)
static int join_context(FmtHandle* h, DevBuf& dst, const float* prev, const float* cur, int C, cudaStream_t st) {
  const ModelShape& s = h->shape;
  const size_t np = static_cast<size_t>(s.P) * C * 4, nl = static_cast<size_t>(s.L) * C * 4;
  FMT_OK(dev_alloc(h, dst, s.B * (np + nl)));
  char* d = static_cast<char*>(dst.p);
  if (np > 0) CUDA_OK(cudaMemcpy2DAsync(d, np + nl, prev, np, np, s.B, cudaMemcpyDeviceToDevice, st));
  CUDA_OK(cudaMemcpy2DAsync(d + np, np + nl, cur, nl, nl, s.B, cudaMemcpyDeviceToDevice, st));
  return 0;
}

template <typename T>
static int enqueue_velocity(FmtHandle* h, const FmtEval* ev, cudaStream_t st) {
  const ModelShape& s = h->shape;
  const GraphShape g = plan_graph(h);
  FMT_OK(enqueue_prepare<T>(h, g, st));
  FMT_OK(enqueue_tables<T>(h, g, ev->eval_index, 1, st));
  const size_t nfull = static_cast<size_t>(s.B) * s.N * s.W;
  FMT_OK(launch(h, init_window_kernel<T>, dim3(static_cast<unsigned>((nfull + 255) / 256)), dim3(256), 0, st, 1,
                static_cast<const WindowArgs*>(h->wargs.p), s, static_cast<float*>(h->xstate.p), static_cast<float*>(h->prevx.p),
                static_cast<T*>(h->ax.p)));
  FMT_OK(enqueue_forward<T>(h, g, 0, st));
  FMT_OK(launch_combine<T>(h, s, 0, ev->v_out, nullptr, st));
  return 0;
}

extern "C" {

int32_t fmt_velocity(FmtHandle* h, const FmtEval* ev, void* stream) {
  REQUIRE(h && ev, "fmt_velocity: null argument");
  REQUIRE(h->configured, "fmt_velocity: call fmt_configure first");
  REQUIRE(ev->eval_index >= 0 && ev->eval_index < h->n_eval, "fmt_velocity: eval_index %d out of range [0,%d)", ev->eval_index, h->n_eval);
  REQUIRE(ev->x && ev->prev_x && ev->wa && ev->prev_wa && ev->we && ev->r_s && ev->v_out, "fmt_velocity: null tensor pointer");
  REQUIRE(!h->plan.we_dynamic || ev->prev_we, "fmt_velocity: dynamic we requires prev_we (FMT.py:306-307)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_OK(cudaSetDevice(h->device));
  const ModelShape& s = h->shape;
  // clip b is slot b: x and its explicit context (init_window_kernel reads ctx, and fmt_velocity runs no finalize_window_kernel that
  // would write it), and [prev | current] frames of its conditions, read from frame P on
  const int NF = s.P + s.L;
  FMT_OK(join_context(h, h->ev_wa, ev->prev_wa, ev->wa, s.A, st));
  const int dyn = h->plan.we_dynamic;
  if (dyn) FMT_OK(join_context(h, h->ev_we, ev->prev_we, ev->we, s.E, st));
  FMT_OK(stage_slot_records(h, 1, false, s.B, st));
  for (int b = 0; b < s.B; ++b) {
    SlotArgs& z = staged_args(h, 0)[b];
    z.r_s = ev->r_s + static_cast<size_t>(b) * s.W;
    z.wa = static_cast<const float*>(h->ev_wa.p) + static_cast<size_t>(b) * NF * s.A;
    z.we = dyn ? static_cast<const float*>(h->ev_we.p) + static_cast<size_t>(b) * NF * s.E : ev->we + static_cast<size_t>(b) * s.E;
    z.x0 = ev->x + static_cast<size_t>(b) * s.L * s.W;
    z.ctx = const_cast<float*>(ev->prev_x) + static_cast<size_t>(b) * s.P * s.W;
    z.T_wa = NF; z.T_we = dyn ? NF : 1; z.we_dynamic = dyn; z.win_start = s.P; z.first_window = 0;
    z.a_scale = ev->a_cfg_scale; z.r_scale = ev->r_cfg_scale; z.e_scale = ev->e_cfg_scale;
  }
  FMT_OK(upload_slot_records(h, 1, st));
  FMT_OK(set_wargs(h, WindowArgs{device_args(h, 0)}, st));
  switch (h->plan.mode) {
    case FMT_MODE_BF16: return enqueue_velocity<bf16>(h, ev, st);
    case FMT_MODE_BF16X3: return enqueue_velocity<bf16x3_t>(h, ev, st);
  }
  return enqueue_velocity<float>(h, ev, st);
}

// ------------------------------------------------------------------------------------------------ diagnostics

// ------------------------------------------------------------------------------------------------ audio projection (SURVEY.md 8f rank 2)
// wa = SiLU(LayerNorm(Linear(wav2vec features)))  -  FLOAT.py:338-342, applied by FloatApplyAudioProjection (nodes_vadv.py:147-198)
struct FmtProj {
  FmtHandle h;            // bare handle: device, SM count, tensor-map encoder, launch counters
  Linear lin;
  float *ln_w = nullptr, *ln_b = nullptr;
  float eps = 1e-5f;
  DevBuf x32, x16, y, o;
};

int32_t fmt_proj_create(int32_t in_dim, int32_t out_dim, const float* w, const float* b, const float* ln_w, const float* ln_b, float ln_eps,
                        int32_t location, int32_t device, FmtProj** out) {
  REQUIRE(w && b && ln_w && ln_b && out, "fmt_proj_create: null argument");
  REQUIRE(in_dim > 0 && in_dim % 16 == 0 && out_dim > 0 && out_dim % 32 == 0, "fmt_proj_create: in_dim %% 16 and out_dim %% 32 required (got %d -> %d)",
          in_dim, out_dim);
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return set_err(-4, "fmt_proj_create: no CUDA device - this library has no CPU fallback");
  REQUIRE(device >= 0 && device < n_dev, "fmt_proj_create: device %d out of range (%d devices)", device, n_dev);
  CUDA_OK(cudaSetDevice(device));
  FmtProj* p = new FmtProj();
  int rc = debug_handle(p->h);
  if (rc == 0) rc = make_linear(&p->h, p->lin, w, b, out_dim, in_dim, in_dim, location);
  if (rc == 0) rc = upload(&p->h, ln_w, out_dim, location, &p->ln_w);
  if (rc == 0) rc = upload(&p->h, ln_b, out_dim, location, &p->ln_b);
  if (rc == 0 && cudaDeviceSynchronize() != cudaSuccess) rc = set_err(-2, "fmt_proj_create: weight packing failed");
  if (rc != 0) { for (void* q : p->h.owned) cudaFree(q); delete p; return rc; }
  p->eps = ln_eps;
  p->h.use_pdl = false;
  *out = p;
  return 0;
}

int32_t fmt_proj_destroy(FmtProj* p) {
  if (!p) return 0;
  cudaSetDevice(p->h.device);
  cudaDeviceSynchronize();
  for (void* q : p->h.owned) cudaFree(q);
  for (DevBuf* bf : {&p->x32, &p->x16, &p->y, &p->o})
    if (bf->p) cudaFree(bf->p);
  delete p;
  return 0;
}

// x: (rows, in_dim) fp32, out: (rows, out_dim) fp32, both at `location`.  FMT_MODE_BF16: bf16 tcgen05 GEMM with fp32 accumulation,
// LayerNorm / SiLU in fp32; FMT_MODE_BF16X3: the split bf16x3 GEMM (in_dim % 64); FMT_MODE_FP32_VALIDATE: fp32 SIMT GEMM.
int32_t fmt_proj_apply(FmtProj* p, const float* x, int64_t rows, float* out, int32_t mode, int32_t location, void* stream) {
  REQUIRE(p && x && out, "fmt_proj_apply: null argument");
  REQUIRE(rows > 0 && rows < (1ll << 31), "fmt_proj_apply: rows = %lld out of range", static_cast<long long>(rows));
  REQUIRE(mode == FMT_MODE_BF16 || mode == FMT_MODE_FP32_VALIDATE || mode == FMT_MODE_BF16X3, "fmt_proj_apply: unknown mode %d", mode);
  FmtHandle* h = &p->h;
  CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int K = p->lin.K, N = p->lin.N, M = static_cast<int>(rows);
  const size_t nx = static_cast<size_t>(rows) * K, ny = static_cast<size_t>(rows) * N;
  const float* xd = x;
  if (location == FMT_LOC_HOST) {
    FMT_OK(dev_alloc(h, p->x32, nx * sizeof(float)));
    CUDA_OK(cudaMemcpyAsync(p->x32.p, x, nx * sizeof(float), cudaMemcpyHostToDevice, st));
    xd = static_cast<const float*>(p->x32.p);
  }
  FMT_OK(dev_alloc(h, p->y, ny * sizeof(float)));
  EpiParams ep = epi(EPI_STORE, M, N, p->lin.b, p->y.p, N, 1);
  if (mode == FMT_MODE_BF16) {
    FMT_OK(dev_alloc(h, p->x16, nx * sizeof(bf16)));
    const size_t n8 = nx / 8;                                   // K % 16 == 0
    const unsigned blocks = static_cast<unsigned>(std::min<size_t>((n8 + 255) / 256, static_cast<size_t>(h->num_sms) * 16));
    f32_to_bf16_kernel<<<blocks, 256, 0, st>>>(xd, static_cast<bf16*>(p->x16.p), n8);
    LAUNCH_CHECK(); count_launch(h);
    FMT_OK(gemm_bf16(h, static_cast<const bf16*>(p->x16.p), K, p->lin.w16, K, ep, K, st));
  } else if (mode == FMT_MODE_BF16X3) {
    REQUIRE(K % 64 == 0, "fmt_proj_apply: bf16x3 mode needs in_dim %% 64 == 0 (got %d)", K);
    FMT_OK(pack_split(h, p->lin, st));
    FMT_OK(dev_alloc(h, p->x16, nx * sizeof(bf16x3_t)));       // x16 holds the GEMM operand of whichever mode ran last
    const size_t n4 = nx / 4;
    const unsigned blocks = static_cast<unsigned>(std::min<size_t>((n4 + 255) / 256, static_cast<size_t>(h->num_sms) * 16));
    f32_to_split_kernel<<<blocks, 256, 0, st>>>(xd, static_cast<bf16x3_t*>(p->x16.p), n4);
    LAUNCH_CHECK(); count_launch(h);
    FMT_OK(gemm_bf16<true>(h, static_cast<const bf16*>(p->x16.p), K, p->lin.w3, K, ep, K, st));
  } else {
    FMT_OK(gemm_f32(h, xd, K, p->lin.w32, K, ep, K, st));
  }
  float* od = out;
  if (location == FMT_LOC_HOST) {
    FMT_OK(dev_alloc(h, p->o, ny * sizeof(float)));
    od = static_cast<float*>(p->o.p);
  }
  const int warps = 8;
  ln_silu_kernel<<<static_cast<unsigned>((rows + warps - 1) / warps), warps * 32, 0, st>>>(static_cast<const float*>(p->y.p), rows, N, p->ln_w, p->ln_b, p->eps, od);
  LAUNCH_CHECK(); count_launch(h);
  if (location == FMT_LOC_HOST) {
    CUDA_OK(cudaMemcpyAsync(out, od, ny * sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
  }
  return 0;
}

int64_t fmt_proj_launch_count(const FmtProj* p, int32_t reset) {
  if (!p) return 0;
  FmtProj* q = const_cast<FmtProj*>(p);
  const long long n = q->h.launches;
  if (reset) q->h.launches = 0;
  return n;
}

int32_t fmt_debug_gemm_bf16(const void* A, const void* W, const float* bias, float* out, int32_t M, int32_t N, int32_t K, int32_t block_n, void* stream) {
  FmtHandle h;
  FMT_OK(debug_handle(h));
  h.use_pdl = false;
  if (const char* e = getenv("FMT_RASTER_GM")) { int v = atoi(e); if (v >= 1) h.raster_gm = v; }
  EpiParams ep = epi(EPI_STORE, M, N, bias, out, N, 1);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return gemm_bf16(&h, static_cast<const bf16*>(A), K, static_cast<const bf16*>(W), K, ep, K, st, block_n);
}

// `iters` back-to-back launches of one bf16 GEMM kernel variant through a single handle (kernel timing in isolation)
int32_t fmt_debug_gemm_bench(const void* A, const void* W, const float* bias, float* out, int32_t M, int32_t N, int32_t K, int32_t block_n,
                             int32_t iters, void* stream) {
  static FmtHandle* hp = nullptr;       // device queries are slow: keep them out of the timed launches
  if (!hp) { hp = new FmtHandle(); FMT_OK(debug_handle(*hp)); }
  FmtHandle& h = *hp;
  h.use_pdl = false;
  if (const char* e = getenv("FMT_RASTER_GM")) { int v = atoi(e); if (v >= 1) h.raster_gm = v; }
  EpiParams ep = epi(EPI_STORE, M, N, bias, out, N, 0);     // bf16 output, like the qkv / fc1 GEMMs of the step
  for (int i = 0; i < iters; ++i)
    FMT_OK(gemm_bf16(&h, static_cast<const bf16*>(A), K, static_cast<const bf16*>(W), K, ep, K, static_cast<cudaStream_t>(stream), block_n));
  return 0;
}

int32_t fmt_debug_gemm_bf16x3(const float* A, const float* W, const float* bias, float* out, int32_t M, int32_t N, int32_t K, int32_t block_n,
                              void* stream) {
  REQUIRE(A && W && out && M > 0 && N > 0 && K > 0 && K % 64 == 0, "fmt_debug_gemm_bf16x3: K %% 64 == 0 and non-null operands required (K=%d)", K);
  FmtHandle h;
  FMT_OK(debug_handle(h));
  h.use_pdl = false;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t na = static_cast<size_t>(M) * K, nw = static_cast<size_t>(N) * K;
  void *a3 = nullptr, *w3 = nullptr;
  CUDA_OK(cudaMallocAsync(&a3, na * sizeof(bf16x3_t), st));
  CUDA_OK(cudaMallocAsync(&w3, nw * sizeof(bf16x3_t), st));
  f32_to_split_kernel<<<static_cast<unsigned>(std::min<size_t>((na / 4 + 255) / 256, 2368)), 256, 0, st>>>(A, static_cast<bf16x3_t*>(a3), na / 4);
  f32_to_split_kernel<<<static_cast<unsigned>(std::min<size_t>((nw / 4 + 255) / 256, 2368)), 256, 0, st>>>(W, static_cast<bf16x3_t*>(w3), nw / 4);
  LAUNCH_CHECK();
  const int rc = gemm_bf16<true>(&h, static_cast<const bf16*>(a3), K, static_cast<const bf16*>(w3), K, epi(EPI_STORE, M, N, bias, out, N, 1), K, st, block_n);
  (void)cudaFreeAsync(a3, st);
  (void)cudaFreeAsync(w3, st);
  return rc;
}

// `iters` back-to-back launches of one bf16x3 GEMM variant on operands already in the pair layout, fp32 output
int32_t fmt_debug_gemm_bench_bf16x3(const void* A, const void* W, const float* bias, float* out, int32_t M, int32_t N, int32_t K, int32_t block_n,
                                    int32_t iters, void* stream) {
  static FmtHandle* hp = nullptr;
  if (!hp) { hp = new FmtHandle(); FMT_OK(debug_handle(*hp)); }
  FmtHandle& h = *hp;
  h.use_pdl = false;
  EpiParams ep = epi(EPI_STORE, M, N, bias, out, N, 1);
  for (int i = 0; i < iters; ++i)
    FMT_OK(gemm_bf16<true>(&h, static_cast<const bf16*>(A), K, static_cast<const bf16*>(W), K, ep, K, static_cast<cudaStream_t>(stream), block_n));
  return 0;
}

int32_t fmt_debug_gemm_fp32(const float* A, const float* W, const float* bias, float* out, int32_t M, int32_t N, int32_t K, void* stream) {
  FmtHandle h;
  EpiParams ep = epi(EPI_STORE, M, N, bias, out, N, 1);
  return gemm_f32(&h, A, K, W, K, ep, K, static_cast<cudaStream_t>(stream));
}

static_assert(FMT_EPI_STORE == int{EPI_STORE} && FMT_EPI_GELU == int{EPI_GELU} && FMT_EPI_POS == int{EPI_POS} && FMT_EPI_GATE_RES == int{EPI_GATE_RES},
              "FMT_EPI_* are the kernels' EpiKind");

int32_t fmt_debug_gemm_epilogue(const FmtDebugGemm* g, void* stream) {
  REQUIRE(g && g->A && g->W && g->out, "fmt_debug_gemm_epilogue: null argument");
  REQUIRE(g->M > 0 && g->N > 0 && g->K > 0 && g->ldo >= g->N, "fmt_debug_gemm_epilogue: bad shape M=%d N=%d K=%d ldo=%d", g->M, g->N, g->K, g->ldo);
  REQUIRE(g->kind >= FMT_EPI_STORE && g->kind <= FMT_EPI_GATE_RES, "fmt_debug_gemm_epilogue: unknown kind %d", g->kind);
  REQUIRE(g->kind != FMT_EPI_POS || (g->pos && g->frames > 0), "fmt_debug_gemm_epilogue: POS needs pos and frames");
  REQUIRE(g->kind != FMT_EPI_GATE_RES || (g->gate && g->out_f32), "fmt_debug_gemm_epilogue: GATE_RES needs a gate table and fp32 out");
  REQUIRE(g->mode == FMT_MODE_BF16 || g->mode == FMT_MODE_FP32_VALIDATE || g->mode == FMT_MODE_BF16X3, "fmt_debug_gemm_epilogue: unknown mode %d", g->mode);
  REQUIRE(g->mode != FMT_MODE_FP32_VALIDATE || (g->block_n == 0 && g->ksplit == 1), "fmt_debug_gemm_epilogue: the fp32 SIMT GEMM has one tile shape");
  REQUIRE(g->mode != FMT_MODE_BF16X3 || g->out_f32 || g->ldo % 64 == 0, "fmt_debug_gemm_epilogue: a pair output needs ldo %% 64 == 0");
  FmtHandle h;
  FMT_OK(debug_handle(h));
  h.use_pdl = false;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  EpiParams ep = epi(g->kind, g->M, g->N, g->bias, g->out, g->ldo, g->out_f32);
  ep.pos = g->pos; ep.frames = g->frames;
  ep.gate = g->gate; ep.urow = g->urow; ep.ldg = g->ldg; ep.gate_off = g->gate_off;
  const int M = g->M, N = g->N, K = g->K;
  if (g->mode == FMT_MODE_FP32_VALIDATE) return gemm_f32(&h, g->A, K, g->W, K, ep, K, st);
  // the operands as the sampler holds them: bf16, or bf16x3 pairs (4 bytes per element either way is enough room)
  const size_t na = static_cast<size_t>(M) * K, nw = static_cast<size_t>(N) * K;
  void *a = nullptr, *w = nullptr;
  CUDA_OK(cudaMallocAsync(&a, na * sizeof(bf16x3_t), st));
  CUDA_OK(cudaMallocAsync(&w, nw * sizeof(bf16x3_t), st));
  int rc = 0;
  if (g->mode == FMT_MODE_BF16) {
    if (K % 8 != 0) rc = set_err(-1, "fmt_debug_gemm_epilogue: K %% 8 required (K=%d)", K);
    if (rc == 0) {
      f32_to_bf16_kernel<<<static_cast<unsigned>(std::min<size_t>((na / 8 + 255) / 256, 2368)), 256, 0, st>>>(g->A, static_cast<bf16*>(a), na / 8);
      f32_to_bf16_kernel<<<static_cast<unsigned>(std::min<size_t>((nw / 8 + 255) / 256, 2368)), 256, 0, st>>>(g->W, static_cast<bf16*>(w), nw / 8);
      rc = cudaGetLastError() == cudaSuccess ? 0 : set_err(-2, "fmt_debug_gemm_epilogue: operand conversion failed");
    }
    if (rc == 0) rc = gemm_bf16(&h, static_cast<const bf16*>(a), K, static_cast<const bf16*>(w), K, ep, K, st, g->block_n, g->ksplit);
  } else {
    if (K % 64 != 0) rc = set_err(-1, "fmt_debug_gemm_epilogue: bf16x3 mode needs K %% 64 == 0 (K=%d)", K);
    if (rc == 0) {
      f32_to_split_kernel<<<static_cast<unsigned>(std::min<size_t>((na / 4 + 255) / 256, 2368)), 256, 0, st>>>(g->A, static_cast<bf16x3_t*>(a), na / 4);
      f32_to_split_kernel<<<static_cast<unsigned>(std::min<size_t>((nw / 4 + 255) / 256, 2368)), 256, 0, st>>>(g->W, static_cast<bf16x3_t*>(w), nw / 4);
      rc = cudaGetLastError() == cudaSuccess ? 0 : set_err(-2, "fmt_debug_gemm_epilogue: operand split failed");
    }
    if (rc == 0) rc = gemm_bf16<true>(&h, static_cast<const bf16*>(a), K, static_cast<const bf16*>(w), K, ep, K, st, g->block_n, g->ksplit);
  }
  (void)cudaFreeAsync(a, st);
  (void)cudaFreeAsync(w, st);
  return rc;
}

int32_t fmt_debug_lnmod(int32_t mode, const float* X, int32_t rows, int32_t H, const void* table, const int32_t* urow, int64_t ldt,
                        int64_t shift_off, int64_t scale_off, void* out, void* stream) {
  REQUIRE(X && table && out && rows > 0, "fmt_debug_lnmod: null argument or no rows");
  FmtHandle h;
  FMT_OK(debug_handle(h));
  h.use_pdl = false;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (mode) {
    case FMT_MODE_BF16: return lnmod<bf16>(&h, X, rows, H, static_cast<const bf16*>(table), urow, ldt, shift_off, scale_off, static_cast<bf16*>(out), st);
    case FMT_MODE_FP32_VALIDATE: return lnmod<float>(&h, X, rows, H, static_cast<const float*>(table), urow, ldt, shift_off, scale_off, static_cast<float*>(out), st);
    case FMT_MODE_BF16X3:
      return lnmod<bf16x3_t>(&h, X, rows, H, static_cast<const float*>(table), urow, ldt, shift_off, scale_off, static_cast<bf16x3_t*>(out), st);
  }
  return set_err(-1, "fmt_debug_lnmod: unknown mode %d", mode);
}

int32_t fmt_debug_band_attention(int32_t mode, const void* qkv, int32_t n_seq, int32_t N, int32_t heads, int32_t hd, int32_t window, void* out,
                                 int32_t variant, void* stream) {
  REQUIRE(qkv && out && n_seq > 0 && N > 0 && heads > 0 && window >= 0, "fmt_debug_band_attention: null argument or bad shape");
  REQUIRE(variant == ATTN_AUTO || variant == ATTN_WARP || variant == ATTN_TILE, "fmt_debug_band_attention: unknown variant %d", variant);
  FmtHandle h;
  FMT_OK(debug_handle(h));
  h.use_pdl = false;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (mode) {
    case FMT_MODE_BF16: return band_attention<bf16>(&h, static_cast<const bf16*>(qkv), n_seq, N, heads, hd, window, static_cast<bf16*>(out), variant, st);
    case FMT_MODE_FP32_VALIDATE:
      return band_attention<float>(&h, static_cast<const float*>(qkv), n_seq, N, heads, hd, window, static_cast<float*>(out), variant, st);
    case FMT_MODE_BF16X3:
      return band_attention<bf16x3_t>(&h, static_cast<const float*>(qkv), n_seq, N, heads, hd, window, static_cast<bf16x3_t*>(out), variant, st);
  }
  return set_err(-1, "fmt_debug_band_attention: unknown mode %d", mode);
}

// ---- row-wise stages of the persistent window kernels
static_assert(FMT_STAGE_ROW == int{FK_ROW} && FMT_STAGE_ATTN == int{FK_ATTN} && FMT_STAGE_GELU == int{FK_GELU} && FMT_STAGE_COMB == int{FK_COMB},
              "FMT_STAGE_* are the kernels' stage kinds");

// Shape and pointer checks shared by both kernels (no device call: bad arguments are refused on any machine)
static int check_stage(const FmtDebugStage* d, const char* fn) {
  REQUIRE(d, "%s: null argument", fn);
  REQUIRE(d->kind >= FMT_STAGE_ROW && d->kind <= FMT_STAGE_COMB, "%s: unknown stage kind %d", fn, d->kind);
  REQUIRE(d->grid >= 0, "%s: grid %d", fn, d->grid);
  REQUIRE(d->H == 128 || d->H == 256 || d->H == 512 || d->H == 1024, "%s: H = %d is not 128, 256, 512 or 1024", fn, d->H);
  REQUIRE(d->n_branches == 1 || d->n_branches == 3 || d->n_branches == 4, "%s: %d CFG branches", fn, d->n_branches);
  REQUIRE(d->batch >= 1 && d->n_frames >= 1 && d->n_prev >= 0 && d->n_prev < d->n_frames, "%s: bad sequence shape batch=%d frames=%d prev=%d", fn,
          d->batch, d->n_frames, d->n_prev);
  if (d->kind == FMT_STAGE_ROW) {
    REQUIRE(d->X && d->Pacc && d->A1 && d->table && d->bias && (d->row_mode == 1 || d->pos), "%s: ROW needs X, Pacc, A1, table, bias (and pos in mode 0)", fn);
    REQUIRE(d->row_mode == 0 || d->row_mode == 1, "%s: row mode %d", fn, d->row_mode);
    REQUIRE(d->shift_off >= 0 && d->scale_off >= 0 && d->gate_off >= 0 && d->ldt % 4 == 0 && d->shift_off % 4 == 0 && d->scale_off % 4 == 0 &&
                d->gate_off % 4 == 0 && d->shift_off + d->H <= d->ldt && d->scale_off + d->H <= d->ldt && d->gate_off + d->H <= d->ldt,
            "%s: table columns outside a row of %lld", fn, static_cast<long long>(d->ldt));
  } else if (d->kind == FMT_STAGE_ATTN) {
    REQUIRE(d->QKVacc && d->A2 && d->bias, "%s: ATTN needs QKVacc, A2 and bias", fn);
    const int hd = d->heads > 0 && d->H % d->heads == 0 ? d->H / d->heads : 0;
    REQUIRE(hd == 32 || hd == 64 || hd == 128, "%s: head_dim %d (H = %d, %d heads) is not 32, 64 or 128", fn, hd, d->H, d->heads);
    REQUIRE(d->window >= 0, "%s: window %d", fn, d->window);
  } else if (d->kind == FMT_STAGE_GELU) {
    REQUIRE(d->Hacc && d->Hm && d->bias, "%s: GELU needs Hacc, Hm and bias", fn);
    REQUIRE(d->mlp_hidden > 0 && d->mlp_hidden % 64 == 0, "%s: mlp_hidden %d is not a multiple of 64", fn, d->mlp_hidden);
  } else {
    REQUIRE(d->Vacc && d->bias && d->x_state && d->ddt && d->ax && (d->n_stages == 1 || d->kbuf), "%s: COMB needs Vacc, bias, x_state, ddt, ax (and kbuf)", fn);
    REQUIRE(d->W > 0 && d->n_stages >= 1 && d->n_stages <= 4 && d->stage >= 0 && d->stage < d->n_stages && d->step >= 0,
            "%s: bad COMB arguments W=%d stages=%d stage=%d step=%d", fn, d->W, d->n_stages, d->stage, d->step);
    REQUIRE(!d->slot_branches == !d->slot_scales, "%s: slot_branches and slot_scales go together", fn);
    for (int b = 0; d->slot_branches && b < d->batch; ++b) {
      const int nb = d->slot_branches[b];
      REQUIRE((nb == 1 || nb == 3 || nb == 4) && nb <= d->n_branches, "%s: clip %d combines %d of %d branches", fn, b, nb, d->n_branches);
    }
  }
  return 0;
}

static ModelShape stage_shape(const FmtDebugStage* d) {
  ModelShape s{};
  s.B = d->batch; s.nb = d->n_branches; s.N = d->n_frames; s.P = d->n_prev; s.L = d->n_frames - d->n_prev; s.W = d->W; s.H = d->H;
  return s;
}

static StageArgs stage_args(const FmtDebugStage* d) {
  StageArgs a{};
  a.kind = d->kind; a.row_mode = d->row_mode; a.zero_qkv = d->zero_qkv; a.parity = d->parity;
  a.gate_off = d->gate_off; a.shift_off = d->shift_off; a.scale_off = d->scale_off;
  a.bias = d->bias; a.step = d->step; a.stage = d->stage;
  return a;
}

// One device buffer: a copy of `head` (WinParams, whose `wargs` field is set here), then the WindowArgs and the SlotArgs of every
// clip, with its guidance (slot_branches / slot_scales, else n_branches and a/r/e_scale); *wargs points at the WindowArgs
static int stage_upload(const FmtDebugStage* d, WinParams* head, cudaStream_t st, void** buf, const WindowArgs** wargs) {
  const size_t head_bytes = head ? sizeof(WinParams) : 0;
  const size_t off = (head_bytes + 255) / 256 * 256;
  std::vector<unsigned char> host(off + sizeof(WindowArgs) + static_cast<size_t>(d->batch) * sizeof(SlotArgs), 0);
  CUDA_OK(cudaMallocAsync(buf, host.size(), st));
  SlotArgs* sl = reinterpret_cast<SlotArgs*>(host.data() + off + sizeof(WindowArgs));
  for (int b = 0; b < d->batch; ++b) {
    const bool own = d->slot_branches != nullptr;
    sl[b].n_branches = own ? d->slot_branches[b] : d->n_branches;
    sl[b].a_scale = own ? d->slot_scales[3 * b] : d->a_scale;
    sl[b].r_scale = own ? d->slot_scales[3 * b + 1] : d->r_scale;
    sl[b].e_scale = own ? d->slot_scales[3 * b + 2] : d->e_scale;
  }
  const WindowArgs wa{reinterpret_cast<const SlotArgs*>(static_cast<unsigned char*>(*buf) + off + sizeof(WindowArgs))};
  memcpy(host.data() + off, &wa, sizeof(WindowArgs));
  *wargs = reinterpret_cast<const WindowArgs*>(static_cast<unsigned char*>(*buf) + off);
  if (head) {
    head->wargs = *wargs;
    memcpy(host.data(), head, head_bytes);
  }
  CUDA_OK(cudaMemcpyAsync(*buf, host.data(), host.size(), cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaStreamSynchronize(st));   // `host` is a stack object
  return 0;
}

int32_t fmt_debug_flow_stage(const FmtDebugStage* d, void* stream) {
  FMT_OK(check_stage(d, "fmt_debug_flow_stage"));
  const int CH = d->chunk_rows;
  REQUIRE(CH == 32 || CH == 64, "fmt_debug_flow_stage: chunk_rows %d is not 32 or 64", CH);
  const int nsub = (d->n_frames + CH - 1) / CH, n_chunks = d->n_branches * d->batch * nsub;
  REQUIRE(n_chunks <= FLOW_MAX_CHUNKS, "fmt_debug_flow_stage: %d chunks > %d", n_chunks, FLOW_MAX_CHUNKS);
  REQUIRE(d->kind != FMT_STAGE_ATTN || d->window <= CH, "fmt_debug_flow_stage: window %d > %d rows per chunk", d->window, CH);
  REQUIRE(d->grid == 0 || d->grid >= n_chunks, "fmt_debug_flow_stage: grid %d < %d chunks", d->grid, n_chunks);
  FmtHandle h;
  FMT_OK(debug_handle(h));
  const int grid = d->grid > 0 ? d->grid : h.num_sms;
  REQUIRE(grid >= n_chunks, "fmt_debug_flow_stage: %d SMs < %d chunks", grid, n_chunks);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  FlowParams fp{};
  fp.s = stage_shape(d); fp.R = d->n_branches * d->batch * d->n_frames;
  fp.heads = d->heads; fp.window = d->window; fp.mlp_hidden = d->mlp_hidden; fp.NT = static_cast<int>(d->ldt);
  fp.n_steps = d->step + 1; fp.n_stages = d->n_stages;
  fp.CH = CH; fp.nsub = nsub; fp.NPs = nsub * CH; fp.n_chunks = n_chunks; fp.RP = n_chunks * CH;
  fp.X = d->X; fp.Pacc = d->Pacc; fp.QKVacc = d->QKVacc; fp.Hacc = d->Hacc; fp.Vacc = d->Vacc;
  fp.A1 = static_cast<bf16*>(d->A1); fp.A2 = static_cast<bf16*>(d->A2); fp.Hm = static_cast<bf16*>(d->Hm); fp.ax = static_cast<bf16*>(d->ax);
  fp.table = static_cast<const bf16*>(d->table); fp.urow = d->urow; fp.pos = d->pos; fp.b_dec = d->bias;
  fp.x_state = d->x_state; fp.kbuf = d->kbuf; fp.ddt = d->ddt;
  for (int i = 0; i < 16; ++i) fp.rk_a[i] = d->rk_a[i];
  for (int i = 0; i < 4; ++i) fp.rk_b[i] = d->rk_b[i];
  fp.spin_limit = h.flow_spin_limit;
  void* buf = nullptr;
  FMT_OK(stage_upload(d, nullptr, st, &buf, &fp.wargs));
  const StageArgs a = stage_args(d);
  switch (d->H / 128) {
    case 1: fmt_flow_stage_kernel<1><<<grid, FLOW_THREADS, 0, st>>>(fp, a); break;
    case 2: fmt_flow_stage_kernel<2><<<grid, FLOW_THREADS, 0, st>>>(fp, a); break;
    case 4: fmt_flow_stage_kernel<4><<<grid, FLOW_THREADS, 0, st>>>(fp, a); break;
    default: fmt_flow_stage_kernel<8><<<grid, FLOW_THREADS, 0, st>>>(fp, a); break;
  }
  const cudaError_t e = cudaGetLastError();
  (void)cudaFreeAsync(buf, st);
  return e == cudaSuccess ? 0 : set_err(-2, "fmt_debug_flow_stage: launch failed: %s", cudaGetErrorString(e));
}

int32_t fmt_debug_window_stage(const FmtDebugStage* d, void* stream) {
  FMT_OK(check_stage(d, "fmt_debug_window_stage"));
  const int R = d->n_branches * d->batch * d->n_frames;
  REQUIRE(R <= 256, "fmt_debug_window_stage: %d token rows > 256", R);
  REQUIRE(d->urow == nullptr, "fmt_debug_window_stage: the window kernel's table has one row per token row (urow must be NULL)");
  FmtHandle h;
  FMT_OK(debug_handle(h));
  const int grid = d->grid > 0 ? d->grid : h.num_sms;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  WinParams wp{};
  wp.s = stage_shape(d); wp.R = R; wp.Rp = (R + 63) / 64 * 64;
  wp.heads = d->heads; wp.window = d->window; wp.mlp_hidden = d->mlp_hidden; wp.NT = static_cast<int>(d->ldt);
  wp.n_steps = d->step + 1; wp.n_stages = d->n_stages;
  wp.X = d->X; wp.Pacc = d->Pacc; wp.QKVacc = d->QKVacc; wp.Hacc = d->Hacc; wp.Vacc = d->Vacc;
  wp.A1 = static_cast<bf16*>(d->A1); wp.A2 = static_cast<bf16*>(d->A2); wp.Hm = static_cast<bf16*>(d->Hm); wp.ax = static_cast<bf16*>(d->ax);
  wp.table = static_cast<const bf16*>(d->table); wp.pos = d->pos; wp.b_dec = d->bias;
  wp.x_state = d->x_state; wp.kbuf = d->kbuf; wp.ddt = d->ddt;
  for (int i = 0; i < 16; ++i) wp.rk_a[i] = d->rk_a[i];
  for (int i = 0; i < 4; ++i) wp.rk_b[i] = d->rk_b[i];
  void* buf = nullptr;
  FMT_OK(stage_upload(d, &wp, st, &buf, &wp.wargs));
  const WinParams* dp = static_cast<const WinParams*>(buf);
  const StageArgs a = stage_args(d);
  switch (d->H / 128) {
    case 1: fmt_window_stage_kernel<1><<<grid, WIN_THREADS, 0, st>>>(dp, a); break;
    case 2: fmt_window_stage_kernel<2><<<grid, WIN_THREADS, 0, st>>>(dp, a); break;
    case 4: fmt_window_stage_kernel<4><<<grid, WIN_THREADS, 0, st>>>(dp, a); break;
    default: fmt_window_stage_kernel<8><<<grid, WIN_THREADS, 0, st>>>(dp, a); break;
  }
  const cudaError_t e = cudaGetLastError();
  (void)cudaFreeAsync(buf, st);
  return e == cudaSuccess ? 0 : set_err(-2, "fmt_debug_window_stage: launch failed: %s", cudaGetErrorString(e));
}

}  // extern "C"
