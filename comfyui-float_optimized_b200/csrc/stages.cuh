// Diagnostic kernels behind fmt_debug_flow_stage / fmt_debug_window_stage: ONE row-wise stage kind of a persistent window kernel,
// run over every chunk (flow.cuh) or every row (window.cuh) by that kernel's own __device__ stage functions, in its thread layout
// and with its chunk / unit / context tables, so that a unit test can compare the stage with an fp64 reference on inputs it built.
// No GEMM runs and nothing waits: a FlowWait with need = 0 passes at once (flow_wait_flag returns for a zero target).
#pragma once
#include "flow.cuh"

namespace fmt {

struct StageArgs {
  int kind;                                 // FK_ROW, FK_ATTN, FK_GELU, FK_COMB
  int row_mode;                             // ROW: 0 = after the x-embedder, 1 = after proj / fc2
  int zero_qkv;                             // ROW, window kernel: zero the QKV accumulator rows too (after proj)
  int parity;                               // ATTN, flow kernel: QKV buffer read; the other one's slices are zeroed
  long long gate_off, shift_off, scale_off; // ROW: AdaLN table columns
  const float* bias;                        // ROW: proj / fc2 / x-embedder bias; ATTN: qkv bias; GELU: fc1 bias
  int step, stage;                          // COMB
};

// Flow kernel layout: 512 threads, warps 8-15 (the SIMT engine: flow_stid(), named barriers 1 and 3+) run the stage under the
// register budget fmt_flow_kernel gives them; warps 0-7 (the GEMM engine's roles) hand their registers back and leave.
template <int NV>
__global__ void __launch_bounds__(FLOW_THREADS, 1) fmt_flow_stage_kernel(const __grid_constant__ FlowParams p, const StageArgs a) {
  __shared__ FlowChunk chunks[FLOW_MAX_CHUNKS];
  __shared__ FlowUnits units[4 * FLOW_MAX_CHUNKS];
  __shared__ float red_smem[8 * 16];
  flow_chunk_tables<NV>(p, chunks, units, gridDim.x, blockIdx.x);
  __syncthreads();
  const int warp = threadIdx.x >> 5;
  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
  } else if (warp < 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 184;");
    const size_t qkv_buf = static_cast<size_t>(p.RP) * 3 * p.s.H;
    const int hd = p.s.H / p.heads;
    for (int c = 0; c < p.n_chunks; ++c) {
      const FlowUnits un = units[a.kind * FLOW_MAX_CHUNKS + c];
      if (un.u0 < 0) continue;
      const FlowChunk ck = chunks[c];
      FlowWait w;
      w.f0 = nullptr; w.stride1 = w.stride2 = 0; w.n = 1; w.need = 0u; w.code = 0;
      w.e = 0; w.si = 0; w.c = c;
      if (a.kind == FK_ROW) {
        flow_row_units<NV>(p, ck, c, un, red_smem, p.table, a.row_mode, a.bias, a.gate_off, a.shift_off, a.scale_off, w);
      } else if (a.kind == FK_ATTN) {
        const float* q = p.QKVacc + a.parity * qkv_buf;
        float* qo = p.QKVacc + (a.parity ^ 1) * qkv_buf;
        if (hd == 128) flow_attn_units<8>(p, ck, c, un, q, qo, a.bias, w);
        else if (hd == 64) flow_attn_units<4>(p, ck, c, un, q, qo, a.bias, w);
        else flow_attn_units<2>(p, ck, c, un, q, qo, a.bias, w);
      } else if (a.kind == FK_GELU) {
        flow_gelu_units(p, ck, c, un, a.bias, w);
      } else {
        flow_simt_wait(p, w);
        for (int u = un.u0; u < un.n_units; u += un.stride) flow_comb_unit(p, ck, u, a.step, a.stage);
      }
      named_bar_sync(1, FLOW_SIMT);
    }
  }
}

// Window kernel layout: 288 threads, WinParams and WinCtx in shared memory (split-K schedule); warps 1-8 run the stage, warp 0
// (the weight producer) leaves.
template <int NV>
__global__ void __launch_bounds__(WIN_THREADS, 1) fmt_window_stage_kernel(const WinParams* __restrict__ pp, const StageArgs a) {
  __shared__ WinParams p;
  __shared__ float red_smem[16];
  __shared__ WinCtx cx;
  {
    const int4* src = reinterpret_cast<const int4*>(pp);
    int4* dst = reinterpret_cast<int4*>(&p);
    for (int i = threadIdx.x; i < static_cast<int>(sizeof(WinParams) / 16); i += WIN_THREADS) dst[i] = src[i];
  }
  __syncthreads();
  if (threadIdx.x == 0) win_ctx<false>(p, cx);
  __syncthreads();
  if (threadIdx.x < 32) return;
  if (a.kind == FK_ROW) win_row_stage<NV>(p, cx, red_smem, p.table, a.row_mode, a.bias, a.gate_off, a.shift_off, a.scale_off, a.zero_qkv != 0);
  else if (a.kind == FK_ATTN) win_attn_dispatch(p, cx, a.bias);
  else if (a.kind == FK_GELU) win_gelu_stage(p, cx, a.bias, 0u);
  else win_comb_stage(p, cx, a.step, a.stage);
}

}  // namespace fmt
