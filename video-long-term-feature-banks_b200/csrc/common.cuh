// Shared helpers of libvlfb (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "vlfb.h"

namespace vlfb {

void set_error(const char* fmt, ...);

#define VLFB_CHECK_ARG(cond)                                                        \
  do {                                                                              \
    if (!(cond)) {                                                                  \
      ::vlfb::set_error("%s:%d: bad argument: %s", __FILE__, __LINE__, #cond);      \
      return VLFB_E_BADARG;                                                         \
    }                                                                               \
  } while (0)

#define VLFB_CHECK_LAUNCH()                                                         \
  do {                                                                              \
    cudaError_t e__ = cudaGetLastError();                                           \
    if (e__ != cudaSuccess) {                                                       \
      ::vlfb::set_error("%s:%d: CUDA: %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
      return VLFB_E_CUDA;                                                           \
    }                                                                               \
  } while (0)

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                   Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Grid for streaming kernels: a multiple of the SM count (148 on B200), capped by the work.
static inline int stream_grid(int64_t work_items, int threads, int per_thread = 1) {
  int64_t blocks = (work_items + (int64_t)threads * per_thread - 1) / ((int64_t)threads * per_thread);
  const int64_t cap = 148 * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// ---- element-level operand semantics (the definition the tensor-core loaders must match) ----
struct Pos4 { int n, t, h, w; };

__device__ __forceinline__ Pos4 decode_pos(int64_t idx, int T, int H, int W) {
  Pos4 p;
  p.w = (int)(idx % W); idx /= W;
  p.h = (int)(idx % H); idx /= H;
  p.t = (int)(idx % T); idx /= T;
  p.n = (int)idx;
  return p;
}

__device__ __forceinline__ void decode_tap(int tap, int kH, int kW, int& kt, int& kh, int& kw) {
  kw = tap % kW; tap /= kW;
  kh = tap % kH; kt = tap / kH;
}

// Value of operand element (row, k) for z-slice `tap_z` (wgrad) and batch `batch`.
__device__ __forceinline__ float operand_elem(const vlfb_operand_t& op, const vlfb_conv_geom_t& g,
                                              int batch, int tap_z, int64_t row, int k) {
  switch (op.kind) {
    case VLFB_OP_DENSE_K:
      return op.ptr[(int64_t)batch * op.batch_stride + row * op.ld + k];
    case VLFB_OP_DENSE_MN:
      return op.ptr[(int64_t)batch * op.batch_stride + (int64_t)k * op.ld + row];
    case VLFB_OP_CONV_K: {
      Pos4 o = decode_pos(row, g.To, g.Ho, g.Wo);
      int tap = k / g.C, c = k % g.C, kt, kh, kw;
      decode_tap(tap, g.kH, g.kW, kt, kh, kw);
      int ti = o.t * g.sT - g.pT + kt * g.dT, hi = o.h * g.sH - g.pH + kh * g.dH,
          wi = o.w * g.sW - g.pW + kw * g.dW;
      if (ti < 0 || ti >= g.T || hi < 0 || hi >= g.H || wi < 0 || wi >= g.W) return 0.f;
      return op.ptr[((((int64_t)o.n * g.T + ti) * g.H + hi) * g.W + wi) * g.C + c];
    }
    case VLFB_OP_DGRAD_K: {
      Pos4 i = decode_pos(row, g.T, g.H, g.W);
      int tap = k / g.Co, c = k % g.Co, kt, kh, kw;
      decode_tap(tap, g.kH, g.kW, kt, kh, kw);
      int a = i.t + g.pT - kt * g.dT, b = i.h + g.pH - kh * g.dH, cc = i.w + g.pW - kw * g.dW;
      if (a < 0 || b < 0 || cc < 0 || a % g.sT || b % g.sH || cc % g.sW) return 0.f;
      int to = a / g.sT, ho = b / g.sH, wo = cc / g.sW;
      if (to >= g.To || ho >= g.Ho || wo >= g.Wo) return 0.f;
      return op.ptr[((((int64_t)i.n * g.To + to) * g.Ho + ho) * g.Wo + wo) * g.Co + c];
    }
    case VLFB_OP_CONV_MN: {   // k = output position, row = (kh*kW+kw)*C + ci, tap_z = kt
      Pos4 o = decode_pos(k, g.To, g.Ho, g.Wo);
      int tap_hw = (int)row / g.C, ci = (int)row % g.C;
      int kt = tap_z, kh = tap_hw / g.kW, kw = tap_hw % g.kW;
      int ti = o.t * g.sT - g.pT + kt * g.dT, hi = o.h * g.sH - g.pH + kh * g.dH,
          wi = o.w * g.sW - g.pW + kw * g.dW;
      if (ti < 0 || ti >= g.T || hi < 0 || hi >= g.H || wi < 0 || wi >= g.W) return 0.f;
      return op.ptr[((((int64_t)o.n * g.T + ti) * g.H + hi) * g.W + wi) * g.C + ci];
    }
    case VLFB_OP_STEM_K: {   // C == 4 (3 + zero pad); k = (kt*kH+kh)*32 + px*4 + ch; op.ld = row pitch in pixels (0 = W)
      Pos4 o = decode_pos(row, g.To, g.Ho, g.Wo);
      int j = k >> 5, e = k & 31, px = e >> 2, ch = e & 3;
      int kt = j / g.kH, kh = j % g.kH;
      int ti = o.t * g.sT - g.pT + kt, hi = o.h * g.sH - g.pH + kh, wi = o.w * g.sW - g.pW + px;
      if (ti < 0 || ti >= g.T || hi < 0 || hi >= g.H || wi < 0 || wi >= g.W) return 0.f;
      const int64_t pitch = op.ld > 0 ? op.ld : g.W;
      return op.ptr[((((int64_t)o.n * g.T + ti) * g.H + hi) * pitch + wi) * 4 + ch];
    }
    case VLFB_OP_STEM_MN: {  // k = output position, row = kh*32 + px*4 + ch, tap_z = kt
      Pos4 o = decode_pos(k, g.To, g.Ho, g.Wo);
      int kh = (int)row >> 5, px = ((int)row & 31) >> 2, ch = (int)row & 3;
      int kt = tap_z;
      int ti = o.t * g.sT - g.pT + kt, hi = o.h * g.sH - g.pH + kh, wi = o.w * g.sW - g.pW + px;
      if (ti < 0 || ti >= g.T || hi < 0 || hi >= g.H || wi < 0 || wi >= g.W) return 0.f;
      const int64_t pitch = op.ld > 0 ? op.ld : g.W;
      return op.ptr[((((int64_t)o.n * g.T + ti) * g.H + hi) * pitch + wi) * 4 + ch];
    }
  }
  return 0.f;
}

__device__ __forceinline__ float round_tf32(float v) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v));
  return __uint_as_float(u);
}

// Epilogue applied to one accumulator value (shared by both GEMM engines).
__device__ __forceinline__ void epilogue_store(const vlfb_gemm_params_t& p, int batch, int tap, int m,
                                               int n, float v, bool first_split = true) {
  v *= p.alpha;
  if (p.col_scale) v *= p.col_scale[n];
  if (p.col_bias && first_split) v += p.col_bias[n];      // split-K: the bias is added by the first K slice only
  if (p.row_scale) v *= p.row_scale[m];
  int64_t off = (int64_t)batch * p.d_batch_stride + (int64_t)tap * p.d_tap_stride + (int64_t)m * p.ldd + n;
  if (p.residual) v += p.residual[off];
  if (p.flags & VLFB_EPI_ACCUM) v += p.d[off];
  if (p.flags & VLFB_EPI_RELU) v = fmaxf(v, 0.f);
  if (p.relu_mask && !(p.relu_mask[off] > 0.f)) v = 0.f;
  if (p.relu_mask_bits && !((p.relu_mask_bits[off >> 5] >> (off & 31)) & 1u)) v = 0.f;
  if (p.flags & VLFB_EPI_TF32) v = round_tf32(v);
  if (p.flags & VLFB_EPI_ATOMIC) atomicAdd(p.d + off, v);
  else p.d[off] = v;
}

int gemm_simt(const vlfb_gemm_params_t& p, cudaStream_t stream);
int relu_bits(const float* x, uint32_t* bits, int64_t n, cudaStream_t stream);     // ops.cu
int gemm_tc(const vlfb_gemm_params_t& p, cudaStream_t stream);
void gemm_tc_plan(const vlfb_gemm_params_t& p, int num_sms, vlfb_gemm_plan_t* out);
size_t gemm_tc_workspace_bytes();
// True when an accumulating product must not be split into K slices that add into D in arrival order (vlfb.h,
// split_k): the one policy both GEMM engines follow (gemm_tc.cu).
bool gemm_fixed_order_split(const vlfb_gemm_params_t& p);
#ifdef VLFB_TRACE
void gemm_tc_set_trace(void* buf);
#endif

}  // namespace vlfb
