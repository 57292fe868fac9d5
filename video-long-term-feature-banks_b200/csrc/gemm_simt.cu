// SIMT fp32 gathered GEMM -- bring-up / on-GPU cross-check engine only (vlfb_set_gemm_backend(1)).
// It evaluates the operand semantics of common.cuh element by element, so it is the
// executable definition the tcgen05 loaders in gemm_tc.cu are tested against.
#include "common.cuh"

namespace vlfb {

namespace {

constexpr int TM = 32, TN = 32, TK = 16;

__global__ void __launch_bounds__(256) gemm_simt_kernel(const vlfb_gemm_params_t p) {
  __shared__ float sa[TK][TM + 1];
  __shared__ float sb[TK][TN + 1];
  const int z = blockIdx.z;
  const int split = z % p.split_k;
  const int zz = z / p.split_k;
  const int batch = (p.taps > 1) ? 0 : zz;
  const int tap = (p.taps > 1) ? zz : 0;
  const int kper = ((p.K + p.split_k - 1) / p.split_k + TK - 1) / TK * TK;
  const int k_begin = split * kper;
  const int k_end = min(p.K, k_begin + kper);
  const int m0 = blockIdx.x * TM, n0 = blockIdx.y * TN;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;   // 16 x 16 threads, 2x2 outputs each
  float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
  for (int k0 = k_begin; k0 < k_end; k0 += TK) {
    for (int i = threadIdx.x; i < TK * TM; i += 256) {
      int kk = i / TM, mm = i % TM;
      int m = m0 + mm, k = k0 + kk;
      sa[kk][mm] = (m < p.M && k < k_end) ? operand_elem(p.a, p.g, batch, tap, m, k) : 0.f;
    }
    for (int i = threadIdx.x; i < TK * TN; i += 256) {
      int kk = i / TN, nn = i % TN;
      int n = n0 + nn, k = k0 + kk;
      sb[kk][nn] = (n < p.N && k < k_end) ? operand_elem(p.b, p.g, batch, tap, n, k) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < TK; ++kk) {
      float a0 = sa[kk][ty], a1 = sa[kk][ty + 16], b0 = sb[kk][tx], b1 = sb[kk][tx + 16];
      acc[0][0] += a0 * b0; acc[0][1] += a0 * b1; acc[1][0] += a1 * b0; acc[1][1] += a1 * b1;
    }
    __syncthreads();
  }
  if (k_begin >= k_end && split > 0) return;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      int m = m0 + ty + 16 * i, n = n0 + tx + 16 * j;
      if (m < p.M && n < p.N) epilogue_store(p, batch, tap, m, n, acc[i][j], split == 0);
    }
}

}  // namespace

int gemm_simt(const vlfb_gemm_params_t& p_in, cudaStream_t stream) {
  vlfb_gemm_params_t p = p_in;
  // "library's choice": K slices that add into D atomically, unless the caller asked for a fixed summation order
  if (p.split_k == 0)
    p.split_k = gemm_fixed_order_split(p_in) ? 1 : (p.K >= 2048 ? (p.K / 1024 < 32 ? p.K / 1024 : 32) : 1);
  dim3 grid(ceil_div(p.M, TM), ceil_div(p.N, TN), (p.taps > 1 ? p.taps : p.batch) * p.split_k);
  launch_k(gemm_simt_kernel, grid, 256, 0, stream, p);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

}  // namespace vlfb
