// Streaming (HBM-bound) kernels of the hot path: pooling, RoIAlign, softmax, LayerNorm,
// elementwise, layout changes, losses, optimizer, fused FBO attention core.
// All activations fp32 channels-last; 128-bit loads/stores wherever the channel extent allows;
// grids are sized in multiples of the 148 SMs (common.cuh: stream_grid).
#include <float.h>

#include "common.cuh"

namespace vlfb {
namespace {

constexpr int TPB = 256;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// Block-wide reductions for <= 1024 threads; `red` is 32 floats of shared memory.
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = (threadIdx.x < (blockDim.x + 31) / 32) ? red[threadIdx.x] : 0.f;
  if (threadIdx.x < 32) r = warp_sum(r);
  if (threadIdx.x == 0) red[0] = r;
  __syncthreads();
  return red[0];
}
__device__ __forceinline__ float block_max(float v, float* red) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = (threadIdx.x < (blockDim.x + 31) / 32) ? red[threadIdx.x] : -FLT_MAX;
  if (threadIdx.x < 32) r = warp_max(r);
  if (threadIdx.x == 0) red[0] = r;
  __syncthreads();
  return red[0];
}

// ------------------------------------------------------------------ AffineNd
__global__ void affine_fwd_k(const float4* __restrict__ x, const float4* __restrict__ s, const float4* __restrict__ b,
                             float4* __restrict__ y, int64_t n4, int c4) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4);
    const float4 v = x[i], sc = s[c];
    float4 o;
    if (b) {
      const float4 bi = b[c];
      o = make_float4(v.x * sc.x + bi.x, v.y * sc.y + bi.y, v.z * sc.z + bi.z, v.w * sc.w + bi.w);
    } else {
      o = make_float4(v.x * sc.x, v.y * sc.y, v.z * sc.z, v.w * sc.w);
    }
    y[i] = o;
  }
}

// ------------------------------------------------------------------ pooling
__global__ void maxpool_fwd_k(const float* __restrict__ x, float* __restrict__ y, int32_t* __restrict__ arg,
                              const vlfb_conv_geom_t g, int64_t total) {
  const int c4 = g.C >> 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4) * 4;
    const Pos4 o = decode_pos(i / c4, g.To, g.Ho, g.Wo);
    float4 best = make_float4(-FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX);
    int4 bi = make_int4(-1, -1, -1, -1);
    for (int kt = 0; kt < g.kT; ++kt) {
      const int t = o.t * g.sT - g.pT + kt;
      if ((unsigned)t >= (unsigned)g.T) continue;
      for (int kh = 0; kh < g.kH; ++kh) {
        const int h = o.h * g.sH - g.pH + kh;
        if ((unsigned)h >= (unsigned)g.H) continue;
        for (int kw = 0; kw < g.kW; ++kw) {
          const int w = o.w * g.sW - g.pW + kw;
          if ((unsigned)w >= (unsigned)g.W) continue;
          const int pos = ((o.n * g.T + t) * g.H + h) * g.W + w;
          const float4 v = *reinterpret_cast<const float4*>(x + (int64_t)pos * g.C + c);
          if (v.x > best.x) { best.x = v.x; bi.x = pos; }
          if (v.y > best.y) { best.y = v.y; bi.y = pos; }
          if (v.z > best.z) { best.z = v.z; bi.z = pos; }
          if (v.w > best.w) { best.w = v.w; bi.w = pos; }
        }
      }
    }
    *reinterpret_cast<float4*>(y + i * 4) = best;
    if (arg) *reinterpret_cast<int4*>(arg + i * 4) = bi;
  }
}

__global__ void maxpool_bwd_k(const float* __restrict__ dy, const int32_t* __restrict__ arg, float* __restrict__ dx,
                              int C, int64_t total) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int pos = arg[i];
    if (pos >= 0) atomicAdd(dx + (int64_t)pos * C + (i % C), dy[i]);
  }
}

// Gather form of the max-pool backward: every INPUT element sums the gradients of the (few) windows that cover it and
// picked it -- each dx element is written exactly once, so there is no zero fill and there are no atomics (the scatter
// form above: fill + one scalar atomic per output element).  Optional fusions for a pool whose input is a conv + ReLU
// output with no other consumer (pool1): `y` = the pool's OUTPUT gives the ReLU-backward mask of the winner
// (y[o] = x[argmax] > 0; a window whose maximum is 0 passes no gradient), `tf32` rounds the result -- dx is then the
// finished gradient operand of the producer's wgrad GEMM.
__global__ void maxpool_bwd_gather_k(const float* __restrict__ dy, const int32_t* __restrict__ arg,
                                     const float* __restrict__ y, float* __restrict__ dx, const vlfb_conv_geom_t g,
                                     int64_t total, int tf32) {
  const int c4 = g.C >> 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4) * 4;
    const int64_t pos64 = i / c4;
    const int pos = (int)pos64;
    const Pos4 p = decode_pos(pos64, g.T, g.H, g.W);
    // windows covering coordinate x: o * s - pad <= x <= o * s - pad + k - 1
    const int t0 = max(0, (p.t + g.pT - g.kT + g.sT) / g.sT), t1 = min(g.To - 1, (p.t + g.pT) / g.sT);
    const int h0 = max(0, (p.h + g.pH - g.kH + g.sH) / g.sH), h1 = min(g.Ho - 1, (p.h + g.pH) / g.sH);
    const int w0 = max(0, (p.w + g.pW - g.kW + g.sW) / g.sW), w1 = min(g.Wo - 1, (p.w + g.pW) / g.sW);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int ot = t0; ot <= t1; ++ot)
      for (int oh = h0; oh <= h1; ++oh)
        for (int ow = w0; ow <= w1; ++ow) {
          const int64_t o = ((((int64_t)p.n * g.To + ot) * g.Ho + oh) * g.Wo + ow) * g.C + c;
          const int4 a = *reinterpret_cast<const int4*>(arg + o);
          float4 d = *reinterpret_cast<const float4*>(dy + o);
          if (y != nullptr) {
            const float4 m = *reinterpret_cast<const float4*>(y + o);
            d.x = m.x > 0.f ? d.x : 0.f; d.y = m.y > 0.f ? d.y : 0.f; d.z = m.z > 0.f ? d.z : 0.f; d.w = m.w > 0.f ? d.w : 0.f;
          }
          if (a.x == pos) acc.x += d.x;
          if (a.y == pos) acc.y += d.y;
          if (a.z == pos) acc.z += d.z;
          if (a.w == pos) acc.w += d.w;
        }
    if (tf32) { acc.x = round_tf32(acc.x); acc.y = round_tf32(acc.y); acc.z = round_tf32(acc.z); acc.w = round_tf32(acc.w); }
    *reinterpret_cast<float4*>(dx + i * 4) = acc;
  }
}

__global__ void avgpool_fwd_k(const float* __restrict__ x, float* __restrict__ y, const vlfb_conv_geom_t g,
                              int64_t total) {
  const int c4 = g.C >> 2;
  const float inv = 1.f / (float)(g.kT * g.kH * g.kW);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4) * 4;
    const Pos4 o = decode_pos(i / c4, g.To, g.Ho, g.Wo);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int kt = 0; kt < g.kT; ++kt)
      for (int kh = 0; kh < g.kH; ++kh)
        for (int kw = 0; kw < g.kW; ++kw) {
          const int t = o.t * g.sT + kt, h = o.h * g.sH + kh, w = o.w * g.sW + kw;
          const int64_t pos = (((int64_t)o.n * g.T + t) * g.H + h) * g.W + w;
          const float4 v = *reinterpret_cast<const float4*>(x + pos * g.C + c);
          acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
    *reinterpret_cast<float4*>(y + i * 4) = make_float4(acc.x * inv, acc.y * inv, acc.z * inv, acc.w * inv);
  }
}

__global__ void avgpool_bwd_k(const float* __restrict__ dy, float* __restrict__ dx, const vlfb_conv_geom_t g,
                              int accumulate, int64_t total) {
  const int c4 = g.C >> 2;
  const float inv = 1.f / (float)(g.kT * g.kH * g.kW);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4) * 4;
    const Pos4 p = decode_pos(i / c4, g.T, g.H, g.W);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    // output windows [o*s, o*s+k) containing p
    for (int to = max(0, (p.t - g.kT + g.sT) / g.sT); to < g.To && to * g.sT <= p.t; ++to) {
      if (p.t - to * g.sT >= g.kT) continue;
      for (int ho = max(0, (p.h - g.kH + g.sH) / g.sH); ho < g.Ho && ho * g.sH <= p.h; ++ho) {
        if (p.h - ho * g.sH >= g.kH) continue;
        for (int wo = max(0, (p.w - g.kW + g.sW) / g.sW); wo < g.Wo && wo * g.sW <= p.w; ++wo) {
          if (p.w - wo * g.sW >= g.kW) continue;
          const int64_t pos = (((int64_t)p.n * g.To + to) * g.Ho + ho) * g.Wo + wo;
          const float4 v = *reinterpret_cast<const float4*>(dy + pos * g.C + c);
          acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
      }
    }
    float4 o = make_float4(acc.x * inv, acc.y * inv, acc.z * inv, acc.w * inv);
    float4* dst = reinterpret_cast<float4*>(dx + i * 4);
    if (accumulate) { const float4 d = *dst; o.x += d.x; o.y += d.y; o.z += d.z; o.w += d.w; }
    *dst = o;
  }
}

// ------------------------------------------------------------------ RoIAlign (legacy Caffe2)
// All index arithmetic uses explicitly rounded fp32 operations in a fixed order so that it is
// bit-identical to oracle/roi_align_np.py.
struct RoiBox { float x1, y1, bin_h, bin_w; int gh, gw, batch; };

__device__ __forceinline__ RoiBox roi_box(const float* __restrict__ roi, float scale, int PH, int PW, int sr) {
  RoiBox b;
  b.batch = (int)roi[0];
  b.x1 = __fmul_rn(roi[1], scale);
  b.y1 = __fmul_rn(roi[2], scale);
  const float x2 = __fmul_rn(roi[3], scale), y2 = __fmul_rn(roi[4], scale);
  const float rw = fmaxf(__fsub_rn(x2, b.x1), 1.f), rh = fmaxf(__fsub_rn(y2, b.y1), 1.f);
  b.bin_h = __fdiv_rn(rh, (float)PH);
  b.bin_w = __fdiv_rn(rw, (float)PW);
  b.gh = sr > 0 ? sr : (int)ceilf(__fdiv_rn(rh, (float)PH));
  b.gw = sr > 0 ? sr : (int)ceilf(__fdiv_rn(rw, (float)PW));
  return b;
}

__device__ __forceinline__ bool roi_sample(const RoiBox& b, int ph, int pw, int iy, int ix, int H, int W,
                                           int pos[4], float w[4]) {
  float y = __fadd_rn(__fadd_rn(b.y1, __fmul_rn((float)ph, b.bin_h)),
                      __fdiv_rn(__fmul_rn(__fadd_rn((float)iy, 0.5f), b.bin_h), (float)b.gh));
  float x = __fadd_rn(__fadd_rn(b.x1, __fmul_rn((float)pw, b.bin_w)),
                      __fdiv_rn(__fmul_rn(__fadd_rn((float)ix, 0.5f), b.bin_w), (float)b.gw));
  if (y < -1.0f || y > (float)H || x < -1.0f || x > (float)W) {
    pos[0] = pos[1] = pos[2] = pos[3] = -1;
    w[0] = w[1] = w[2] = w[3] = 0.f;
    return false;
  }
  if (y <= 0.f) y = 0.f;
  if (x <= 0.f) x = 0.f;
  int yl = (int)y, xl = (int)x, yh, xh;
  if (yl >= H - 1) { yh = yl = H - 1; y = (float)yl; } else yh = yl + 1;
  if (xl >= W - 1) { xh = xl = W - 1; x = (float)xl; } else xh = xl + 1;
  const float ly = __fsub_rn(y, (float)yl), lx = __fsub_rn(x, (float)xl);
  const float hy = __fsub_rn(1.f, ly), hx = __fsub_rn(1.f, lx);
  w[0] = __fmul_rn(hy, hx); w[1] = __fmul_rn(hy, lx); w[2] = __fmul_rn(ly, hx); w[3] = __fmul_rn(ly, lx);
  pos[0] = yl * W + xl; pos[1] = yl * W + xh; pos[2] = yh * W + xl; pos[3] = yh * W + xh;
  return true;
}

__global__ void roi_align_fwd_k(const float* __restrict__ feat, const float* __restrict__ rois, float* __restrict__ out,
                                int H, int W, int C, int PH, int PW, float scale, int sr, int64_t total) {
  const int c4 = C >> 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4) * 4;
    int64_t q = i / c4;
    const int pw = (int)(q % PW); q /= PW;
    const int ph = (int)(q % PH); q /= PH;
    const int r = (int)q;
    const RoiBox b = roi_box(rois + r * 5, scale, PH, PW, sr);
    const float* f = feat + (int64_t)b.batch * H * W * C + c;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int iy = 0; iy < b.gh; ++iy)
      for (int ix = 0; ix < b.gw; ++ix) {
        int pos[4];
        float w[4];
        if (!roi_sample(b, ph, pw, iy, ix, H, W, pos, w)) continue;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 v = *reinterpret_cast<const float4*>(f + (int64_t)pos[k] * C);
          acc.x += w[k] * v.x; acc.y += w[k] * v.y; acc.z += w[k] * v.z; acc.w += w[k] * v.w;
        }
      }
    const float cnt = (float)(b.gh * b.gw);
    *reinterpret_cast<float4*>(out + i * 4) = make_float4(acc.x / cnt, acc.y / cnt, acc.z / cnt, acc.w / cnt);
  }
}

// Weight that the samples i = 0..g-1 of bin p along one axis (start s, bin size `bin`, extent L) give pixel P: the
// bilinear weights of roi_sample along that axis, zero for a sample outside [-1, L].  A sample's weight at a pixel is
// the product of its two axis weights, and it is dropped when either coordinate is out of range, so the weight of bin
// (ph, pw) at pixel (Y, X) is axis_w(y ..., ph, Y) * axis_w(x ..., pw, X).
__device__ __forceinline__ float roi_axis_w(float s, float bin, int g, int p, int L, int P) {
  float t = 0.f;
  for (int i = 0; i < g; ++i) {
    float v = __fadd_rn(__fadd_rn(s, __fmul_rn((float)p, bin)), __fdiv_rn(__fmul_rn(__fadd_rn((float)i, 0.5f), bin), (float)g));
    if (v < -1.0f || v > (float)L) continue;
    if (v <= 0.f) v = 0.f;
    int lo = (int)v, hi;
    if (lo >= L - 1) { hi = lo = L - 1; v = (float)lo; } else hi = lo + 1;
    const float l = __fsub_rn(v, (float)lo);
    if (lo == P) t += __fsub_rn(1.f, l);
    if (hi == P) t += l;
  }
  return t;
}

constexpr int ROI_BWD_MAX_PW = 32;     // pooled width bound of the backward (x weights of one RoI kept per thread)

// dfeat += RoIAlign backward, gather form: one thread per (image, pixel, 4 channels) sums the contributions of every
// RoI bin in a fixed order and writes its own element once -- no atomics, so the result is the same in every run.
__global__ void roi_align_bwd_k(const float* __restrict__ dout, const float* __restrict__ rois, float* __restrict__ dfeat,
                                int H, int W, int C, int R, int PH, int PW, float scale, int sr, int64_t total) {
  const int c4 = C >> 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4) * 4;
    int64_t q = i / c4;
    const int X = (int)(q % W); q /= W;
    const int Y = (int)(q % H);
    const int n = (int)(q / H);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    bool any = false;
    float wxs[ROI_BWD_MAX_PW];
    for (int r = 0; r < R; ++r) {
      const RoiBox b = roi_box(rois + r * 5, scale, PH, PW, sr);
      if (b.batch != n) continue;
      const float cnt = (float)(b.gh * b.gw);
      bool xhit = false;
      for (int pw = 0; pw < PW; ++pw) {
        wxs[pw] = roi_axis_w(b.x1, b.bin_w, b.gw, pw, W, X);
        xhit |= wxs[pw] != 0.f;
      }
      if (!xhit) continue;
      for (int ph = 0; ph < PH; ++ph) {
        const float wy = roi_axis_w(b.y1, b.bin_h, b.gh, ph, H, Y);
        if (wy == 0.f) continue;
        for (int pw = 0; pw < PW; ++pw) {
          const float wx = wxs[pw];
          if (wx == 0.f) continue;
          const float w = wy * wx / cnt;
          const float4 g = *reinterpret_cast<const float4*>(dout + (((int64_t)r * PH + ph) * PW + pw) * C + c);
          acc.x += w * g.x; acc.y += w * g.y; acc.z += w * g.z; acc.w += w * g.w;
          any = true;
        }
      }
    }
    if (any) {
      float4* d = reinterpret_cast<float4*>(dfeat + (((int64_t)n * H + Y) * W + X) * C + c);
      float4 o = *d;
      o.x += acc.x; o.y += acc.y; o.z += acc.z; o.w += acc.w;
      *d = o;
    }
  }
}

__global__ void roi_table_k(const float* __restrict__ rois, int32_t* __restrict__ pos, float* __restrict__ wts,
                            int32_t* __restrict__ grid, int H, int W, int R, int PH, int PW, int mg, float scale,
                            int sr) {
  const int64_t total = (int64_t)R * PH * PW * mg * mg;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t q = i;
    const int ix = (int)(q % mg); q /= mg;
    const int iy = (int)(q % mg); q /= mg;
    const int pw = (int)(q % PW); q /= PW;
    const int ph = (int)(q % PH); q /= PH;
    const int r = (int)q;
    const RoiBox b = roi_box(rois + r * 5, scale, PH, PW, sr);
    if (ph == 0 && pw == 0 && iy == 0 && ix == 0) { grid[r * 2] = b.gh; grid[r * 2 + 1] = b.gw; }
    int p[4] = {-1, -1, -1, -1};
    float w[4] = {0.f, 0.f, 0.f, 0.f};
    if (iy < b.gh && ix < b.gw) roi_sample(b, ph, pw, iy, ix, H, W, p, w);
#pragma unroll
    for (int k = 0; k < 4; ++k) { pos[i * 4 + k] = p[k]; wts[i * 4 + k] = w[k]; }
  }
}

// ------------------------------------------------------------------ softmax / layernorm (warp per row)
__global__ void softmax_fwd_k(const float* __restrict__ x, float* __restrict__ p, int64_t rows, int cols, float scale,
                              int tf32) {
  const int lane = threadIdx.x & 31;
  const int64_t wpb = blockDim.x >> 5;
  for (int64_t row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += (int64_t)gridDim.x * wpb) {
    const float* xr = x + row * cols;
    float* pr = p + row * cols;
    float mx = -FLT_MAX;
    for (int c = lane; c < cols; c += 32) mx = fmaxf(mx, xr[c] * scale);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int c = lane; c < cols; c += 32) sum += __expf(xr[c] * scale - mx);
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    for (int c = lane; c < cols; c += 32) {
      const float v = __expf(xr[c] * scale - mx) * inv;
      pr[c] = tf32 ? round_tf32(v) : v;
    }
  }
}

__global__ void softmax_bwd_k(const float* __restrict__ p, const float* __restrict__ dp, float* __restrict__ dx,
                              int64_t rows, int cols, float scale, int tf32) {
  const int lane = threadIdx.x & 31;
  const int64_t wpb = blockDim.x >> 5;
  for (int64_t row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += (int64_t)gridDim.x * wpb) {
    const float* pr = p + row * cols;
    const float* dr = dp + row * cols;
    float dot = 0.f;
    for (int c = lane; c < cols; c += 32) dot += pr[c] * dr[c];
    dot = warp_sum(dot);
    for (int c = lane; c < cols; c += 32) {
      const float v = scale * pr[c] * (dr[c] - dot);
      dx[row * cols + c] = tf32 ? round_tf32(v) : v;
    }
  }
}

__global__ void layernorm_fwd_k(const float* __restrict__ x, float* __restrict__ y, float* __restrict__ mean,
                                float* __restrict__ sd, int64_t rows, int cols, float eps) {
  const int lane = threadIdx.x & 31;
  const int64_t wpb = blockDim.x >> 5;
  for (int64_t row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += (int64_t)gridDim.x * wpb) {
    const float* xr = x + row * cols;
    float s = 0.f;
    for (int c = lane; c < cols; c += 32) s += xr[c];
    const float mu = warp_sum(s) / cols;
    float v = 0.f;
    for (int c = lane; c < cols; c += 32) { const float d = xr[c] - mu; v += d * d; }
    const float sdev = sqrtf(warp_sum(v) / cols + eps);
    for (int c = lane; c < cols; c += 32) y[row * cols + c] = (xr[c] - mu) / sdev;
    if (lane == 0) { if (mean) mean[row] = mu; if (sd) sd[row] = sdev; }
  }
}

__global__ void layernorm_bwd_k(const float* __restrict__ dy, const float* __restrict__ y, const float* __restrict__ sd,
                                float* __restrict__ dx, int64_t rows, int cols) {
  const int lane = threadIdx.x & 31;
  const int64_t wpb = blockDim.x >> 5;
  for (int64_t row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += (int64_t)gridDim.x * wpb) {
    const float* dr = dy + row * cols;
    const float* yr = y + row * cols;
    float a = 0.f, b = 0.f;
    for (int c = lane; c < cols; c += 32) { a += dr[c]; b += dr[c] * yr[c]; }
    a = warp_sum(a) / cols;
    b = warp_sum(b) / cols;
    const float inv = 1.f / sd[row];
    for (int c = lane; c < cols; c += 32) dx[row * cols + c] = inv * (dr[c] - a - yr[c] * b);
  }
}

// ------------------------------------------------------------------ elementwise
enum { EW_RELU = 0, EW_RELU_BWD = 1, EW_AXPBY = 2, EW_FILL = 3, EW_SIGMOID = 4, EW_TF32 = 5, EW_ADD_TF32 = 6, EW_RELU_TF32 = 7, EW_RELU_BWD_TF32 = 8 };

template <int OP>
__device__ __forceinline__ float ew_op(float a, float b, float s0, float s1) {
  if (OP == EW_RELU) return fmaxf(a, 0.f);
  if (OP == EW_RELU_BWD) return b > 0.f ? a : 0.f;           // a = dy, b = y
  if (OP == EW_AXPBY) return s0 * a + s1 * b;
  if (OP == EW_FILL) return s0;
  if (OP == EW_TF32) return round_tf32(a);
  if (OP == EW_ADD_TF32) return round_tf32(a + b);
  if (OP == EW_RELU_TF32) return round_tf32(fmaxf(a, 0.f));
  if (OP == EW_RELU_BWD_TF32) return b > 0.f ? round_tf32(a) : 0.f;
  return 1.f / (1.f + __expf(-a));
}

template <int OP>
__global__ void ew_k(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ o, int64_t n,
                     float s0, float s1, int vec) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (vec) {
    const int64_t n4 = n >> 2;
    for (int64_t i = t; i < n4; i += stride) {
      float4 va = a ? reinterpret_cast<const float4*>(a)[i] : make_float4(0, 0, 0, 0);
      float4 vb = b ? reinterpret_cast<const float4*>(b)[i] : make_float4(0, 0, 0, 0);
      reinterpret_cast<float4*>(o)[i] = make_float4(ew_op<OP>(va.x, vb.x, s0, s1), ew_op<OP>(va.y, vb.y, s0, s1),
                                                    ew_op<OP>(va.z, vb.z, s0, s1), ew_op<OP>(va.w, vb.w, s0, s1));
    }
    for (int64_t i = (n4 << 2) + t; i < n; i += stride) o[i] = ew_op<OP>(a ? a[i] : 0.f, b ? b[i] : 0.f, s0, s1);
  } else {
    for (int64_t i = t; i < n; i += stride) o[i] = ew_op<OP>(a ? a[i] : 0.f, b ? b[i] : 0.f, s0, s1);
  }
}

template <int OP>
int ew_launch(const float* a, const float* b, float* o, int64_t n, float s0, float s1, cudaStream_t st) {
  if (n <= 0) return VLFB_OK;
  const bool vec = ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(o)) & 15) == 0;
  launch_k(ew_k<OP>, stream_grid(n, TPB, 4), TPB, 0, st, a, b, o, n, s0, s1, vec ? 1 : 0);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

// out = (y == nullptr || y > 0) ? round_tf32(a + b) : 0 -- the sum of two gradient contributions, the ReLU backward
// of the layer that owns the gradient and the TF32 rounding its GEMMs need, in ONE pass (4 tensor streams instead
// of the 6 of axpby + relu_bwd_tf32).  `out` may alias a or b.
__global__ void add_mask_tf32_k(const float* a, const float* b, const float* y, float* o, int64_t n, int vec) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (vec) {
    const int64_t n4 = n >> 2;
    for (int64_t i = t; i < n4; i += stride) {
      const float4 va = reinterpret_cast<const float4*>(a)[i], vb = reinterpret_cast<const float4*>(b)[i];
      const float4 vy = y ? reinterpret_cast<const float4*>(y)[i] : make_float4(1.f, 1.f, 1.f, 1.f);
      reinterpret_cast<float4*>(o)[i] =
          make_float4(vy.x > 0.f ? round_tf32(va.x + vb.x) : 0.f, vy.y > 0.f ? round_tf32(va.y + vb.y) : 0.f,
                      vy.z > 0.f ? round_tf32(va.z + vb.z) : 0.f, vy.w > 0.f ? round_tf32(va.w + vb.w) : 0.f);
    }
    for (int64_t i = (n4 << 2) + t; i < n; i += stride) o[i] = (!y || y[i] > 0.f) ? round_tf32(a[i] + b[i]) : 0.f;
  } else {
    for (int64_t i = t; i < n; i += stride) o[i] = (!y || y[i] > 0.f) ? round_tf32(a[i] + b[i]) : 0.f;
  }
}

// Philox4x32-10 counter-based generator (Salmon et al. 2011), self-contained.
__device__ __forceinline__ uint4 philox4x32(uint64_t ctr, uint64_t key) {
  uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = 0u, c3 = 0u;
  uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = h1 ^ c1 ^ k0, n1 = l1, n2 = h0 ^ c3 ^ k1, n3 = l0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

__global__ void dropout_k(const float* __restrict__ x, float* __restrict__ y, int64_t n, float ratio, float inv_keep,
                          uint64_t seed, uint64_t offset, const int64_t* __restrict__ step) {
  const int64_t n4 = (n + 3) >> 2;
  if (step) offset += (uint64_t)step[0] << 32;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 r = philox4x32(offset + (uint64_t)i, seed);
    const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int64_t j = i * 4 + e;
      if (j < n) {
        const float u = (float)(rr[e] >> 8) * (1.0f / 16777216.0f);
        y[j] = (u >= ratio) ? x[j] * inv_keep : 0.f;
      }
    }
  }
}

__global__ void copy2d_k(const float* __restrict__ src, int64_t lds, float* __restrict__ dst, int64_t ldd, int64_t rows,
                         int cols, int accumulate) {
  const int64_t total = rows * cols;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols;
    const int c = (int)(i - r * cols);
    const float v = src[r * lds + c];
    if (accumulate) dst[r * ldd + c] += v; else dst[r * ldd + c] = v;
  }
}

// out[c] (+)= sum_r x[r*ld+c]: block = 32 columns x 8 row-lanes over a slab of rows.  With one slab the block writes
// out; otherwise each slab's sums go to part[slab][c] and colsum_finish_k adds the slabs in slab order, so the result
// does not depend on the order in which blocks finish (atomics would make it differ from run to run).
__global__ void colsum_k(const float* __restrict__ x, int64_t ld, float* __restrict__ out, int64_t rows, int cols,
                         int64_t rows_per_block, float* __restrict__ part, int accumulate) {
  __shared__ float sp[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
  const int64_t r1 = min(rows, r0 + rows_per_block);
  float s = 0.f;
  if (c < cols)
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) s += x[r * ld + c];
  sp[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && c < cols) {
    float t = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) t += sp[j][threadIdx.x];
    if (part) part[(int64_t)blockIdx.y * cols + c] = t;
    else out[c] = accumulate ? out[c] + t : t;
  }
}

__global__ void colsum_finish_k(const float* __restrict__ part, int slabs, float* __restrict__ out, int cols,
                                int accumulate) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  float t = 0.f;
  for (int j = 0; j < slabs; ++j) t += part[(int64_t)j * cols + c];
  out[c] = accumulate ? out[c] + t : t;
}

// ------------------------------------------------------------------ layouts
// src [N][C][inner] <-> dst [N][inner][Cpad]; tiled 32x32 transposes through shared memory.
// Clip feeding (C <= 4 planes -> 4-channel pixels): one thread converts 4 consecutive positions: C coalesced 16-byte
// plane loads -> four 16-byte pixel stores (64 contiguous bytes per thread), optional TF32 rounding of the conv1 operand.
// The generic 32x32 tile kernel below moves only 3 of its 32 tile rows for a clip (0.39 TB/s measured).
__global__ void nc_to_cl4_k(const float* __restrict__ src, float4* __restrict__ dst, int C, int64_t inner4,
                            int64_t total, int tf32) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = q / inner4, i4 = q - n * inner4;
    float4 p[4];
#pragma unroll
    for (int c = 0; c < 4; ++c)
      p[c] = c < C ? *reinterpret_cast<const float4*>(src + ((n * C + c) * inner4 + i4) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (tf32) {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        p[c].x = round_tf32(p[c].x); p[c].y = round_tf32(p[c].y); p[c].z = round_tf32(p[c].z); p[c].w = round_tf32(p[c].w);
      }
    }
    float4* o = dst + (n * inner4 + i4) * 4;
    o[0] = make_float4(p[0].x, p[1].x, p[2].x, p[3].x);
    o[1] = make_float4(p[0].y, p[1].y, p[2].y, p[3].y);
    o[2] = make_float4(p[0].z, p[1].z, p[2].z, p[3].z);
    o[3] = make_float4(p[0].w, p[1].w, p[2].w, p[3].w);
  }
}

// ... into rows of `pitch` pixels starting at pixel `left` (W4 = W / 4 groups of 4 pixels per row)
__global__ void nc_to_cl4p_k(const float* __restrict__ src, float4* __restrict__ dst, int C, int64_t inner4, int64_t total,
                             int tf32, int W4, int pitch, int left) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = q / inner4, i4 = q - n * inner4;
    float4 p[4];
#pragma unroll
    for (int c = 0; c < 4; ++c)
      p[c] = c < C ? *reinterpret_cast<const float4*>(src + ((n * C + c) * inner4 + i4) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (tf32) {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        p[c].x = round_tf32(p[c].x); p[c].y = round_tf32(p[c].y); p[c].z = round_tf32(p[c].z); p[c].w = round_tf32(p[c].w);
      }
    }
    const int64_t row = (n * inner4 + i4) / W4;
    const int w4 = (int)((n * inner4 + i4) - row * W4);
    float4* o = dst + row * pitch + left + w4 * 4;
    o[0] = make_float4(p[0].x, p[1].x, p[2].x, p[3].x);
    o[1] = make_float4(p[0].y, p[1].y, p[2].y, p[3].y);
    o[2] = make_float4(p[0].z, p[1].z, p[2].z, p[3].z);
    o[3] = make_float4(p[0].w, p[1].w, p[2].w, p[3].w);
  }
}

__global__ void nc_to_cl_k(const float* __restrict__ src, float* __restrict__ dst, int C, int64_t inner, int Cpad,
                           int tf32) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const int64_t i0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int c = c0 + r;
    const int64_t i = i0 + threadIdx.x;
    tile[r][threadIdx.x] = (c < C && i < inner) ? src[((int64_t)n * C + c) * inner + i] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int64_t i = i0 + r;
    const int c = c0 + threadIdx.x;
    if (i < inner && c < Cpad) {
      const float v = tile[threadIdx.x][r];
      dst[((int64_t)n * inner + i) * Cpad + c] = tf32 ? round_tf32(v) : v;
    }
  }
}

__global__ void cl_to_nc_k(const float* __restrict__ src, float* __restrict__ dst, int C, int64_t inner, int Cpad) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const int64_t i0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int64_t i = i0 + r;
    const int c = c0 + threadIdx.x;
    tile[r][threadIdx.x] = (i < inner && c < C) ? src[((int64_t)n * inner + i) * Cpad + c] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int c = c0 + r;
    const int64_t i = i0 + threadIdx.x;
    if (c < C && i < inner) dst[((int64_t)n * C + c) * inner + i] = tile[threadIdx.x][r];
  }
}

// wt[ci][tap][co] = w[co][tap][ci] * scale[co]
__global__ void weight_transpose_k(const float* __restrict__ w, float* __restrict__ wt, const float* __restrict__ scale,
                                   int Co, int taps, int Ci) {
  __shared__ float tile[32][33];
  const int tap = blockIdx.z;
  const int ci0 = blockIdx.x * 32, co0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int co = co0 + r, ci = ci0 + threadIdx.x;
    float v = 0.f;
    if (co < Co && ci < Ci) {
      v = w[((int64_t)co * taps + tap) * Ci + ci];
      if (scale) v *= scale[co];
    }
    tile[r][threadIdx.x] = v;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int ci = ci0 + r, co = co0 + threadIdx.x;
    if (ci < Ci && co < Co) wt[((int64_t)ci * taps + tap) * Co + co] = round_tf32(tile[threadIdx.x][r]);
  }
}

// the same for every convolution of the net in one launch (block -> job by binary search over block_begin)
__global__ void weight_transpose_multi_k(const vlfb_wt_job_t* __restrict__ jobs, int njobs) {
  __shared__ float tile[32][33];
  // block -> job: the table's block_begin column is fetched by ONE coalesced load into shared memory and searched
  // there (the search over global memory was ~6 dependent L2 round trips per 4 KB tile: call J, 185 us for 238 MB)
  __shared__ int begins[256];
  const int tid = threadIdx.y * 32 + threadIdx.x;
  const bool in_smem = njobs <= 256;
  if (in_smem) {
    if (tid < njobs) begins[tid] = jobs[tid].block_begin;
    __syncthreads();
  }
  int lo = 0, hi = njobs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    const int bb = in_smem ? begins[mid] : jobs[mid].block_begin;
    if (bb <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const vlfb_wt_job_t jb = jobs[lo];
  const int local = blockIdx.x - jb.block_begin;
  const int tci = (jb.Ci + 31) >> 5, tco = (jb.Co + 31) >> 5;
  const int ci0 = (local % tci) * 32, co0 = ((local / tci) % tco) * 32, tap = local / (tci * tco);
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int co = co0 + r, ci = ci0 + threadIdx.x;
    float v = 0.f;
    if (co < jb.Co && ci < jb.Ci) {
      v = jb.w[((int64_t)co * jb.taps + tap) * jb.Ci + ci];
      if (jb.scale) v *= jb.scale[co];
    }
    tile[r][threadIdx.x] = v;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int ci = ci0 + r, co = co0 + threadIdx.x;
    if (ci < jb.Ci && co < jb.Co) jb.wt[((int64_t)ci * jb.taps + tap) * jb.Co + co] = round_tf32(tile[threadIdx.x][r]);
  }
}

// ------------------------------------------------------------------ losses (single block; R*classes is small)
__device__ __forceinline__ float sce_elem(float x, float t) {
  // -(x*(t-(x>=0)) - log(1+exp(x-2x(x>=0))))
  const float ge = x >= 0.f ? 1.f : 0.f;
  return -(x * (t - ge) - log1pf(__expf(x - 2.f * x * ge)));
}

__global__ void sigmoid_ce_fwd_k(const float* __restrict__ x, const int32_t* __restrict__ t, float* __restrict__ loss,
                                 int64_t n, float scale) {
  __shared__ float red[32];
  float s = 0.f, cnt = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const int ti = t[i];
    if (ti != -1) { s += sce_elem(x[i], (float)ti); cnt += 1.f; }
  }
  s = block_sum(s, red);
  cnt = block_sum(cnt, red);
  if (threadIdx.x == 0) loss[0] = scale * s / fmaxf(cnt, 1e-5f);
}

__global__ void sigmoid_ce_bwd_k(const float* __restrict__ x, const int32_t* __restrict__ t,
                                 const float* __restrict__ dloss, float* __restrict__ dx, int64_t n, float scale) {
  __shared__ float red[32];
  float cnt = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) cnt += (t[i] != -1) ? 1.f : 0.f;
  cnt = block_sum(cnt, red);
  const float k = scale / fmaxf(cnt, 1e-5f) * (dloss ? dloss[0] : 1.f);
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const int ti = t[i];
    dx[i] = (ti != -1) ? k * (1.f / (1.f + __expf(-x[i])) - (float)ti) : 0.f;
  }
}

__global__ void softmax_ce_fwd_k(const float* __restrict__ x, const int32_t* __restrict__ lab, float* __restrict__ prob,
                                 float* __restrict__ loss, int rows, int cols, float scale) {
  __shared__ float red[32];
  float total = 0.f;
  for (int r = 0; r < rows; ++r) {
    const float* xr = x + (int64_t)r * cols;
    float mx = -FLT_MAX;
    for (int c = threadIdx.x; c < cols; c += blockDim.x) mx = fmaxf(mx, xr[c]);
    mx = block_max(mx, red);
    float s = 0.f;
    for (int c = threadIdx.x; c < cols; c += blockDim.x) s += __expf(xr[c] - mx);
    s = block_sum(s, red);
    for (int c = threadIdx.x; c < cols; c += blockDim.x) prob[(int64_t)r * cols + c] = __expf(xr[c] - mx) / s;
    total += -(xr[lab[r]] - mx - __logf(s));
  }
  if (threadIdx.x == 0) loss[0] = scale * total / rows;
}

__global__ void softmax_ce_bwd_k(const float* __restrict__ prob, const int32_t* __restrict__ lab, float* __restrict__ dx,
                                 int rows, int cols, float scale) {
  const int64_t total = (int64_t)rows * cols;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    dx[i] = (prob[i] - (c == lab[r] ? 1.f : 0.f)) * scale / rows;
  }
}

// ------------------------------------------------------------------ optimizer
__global__ void sgd_k(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m, float* __restrict__ pt, int64_t n,
                      const float* __restrict__ lrp, float mom, float wd, int nesterov) {
  const float lr = lrp[0];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float pi = p[i], mi = m[i];
    const float gi = g[i] + wd * pi;                       // WeightedSum([g, ONE, p, wd])
    const float mn = mom * mi + lr * gi;                   // MomentumSGDUpdate
    const float ng = nesterov ? (1.f + mom) * mn - mom * mi : mn;
    m[i] = mn;
    g[i] = ng;
    p[i] = pi - ng;
    if (pt) pt[i] = round_tf32(pi - ng);
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// ReLU sign bits: word w = ballot of x[32 w + lane] > 0 (the layout vlfb_gemm_params_t.relu_mask_bits reads).
__global__ void relu_bits_k(const float* __restrict__ x, uint32_t* __restrict__ bits, int64_t words) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t w = warp0; w < words; w += nwarps) {
    const unsigned b = __ballot_sync(0xffffffffu, x[w * 32 + lane] > 0.f);
    if (lane == 0) bits[w] = b;
  }
}

int relu_bits(const float* x, uint32_t* bits, int64_t n, cudaStream_t stream) {
  if (n == 0) return VLFB_OK;
  launch_k(relu_bits_k, stream_grid(n, TPB), TPB, 0, stream, x, bits, n >> 5);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

}  // namespace vlfb

using namespace vlfb;
#define ST(s) static_cast<cudaStream_t>(s)

extern "C" {

int vlfb_affine_nd_fwd(const float* x, const float* scale, const float* bias, float* y, int64_t rows, int C,
                       void* stream) {
  VLFB_CHECK_ARG(x && scale && bias && y && rows >= 0 && C > 0 && (C & 3) == 0);
  const int64_t n4 = rows * (C >> 2);
  if (n4 == 0) return VLFB_OK;
  launch_k(affine_fwd_k, stream_grid(n4, TPB), TPB, 0, ST(stream), (const float4*)x, (const float4*)scale, (const float4*)bias,
                                                             (float4*)y, n4, C >> 2);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_affine_nd_bwd(const float* dy, const float* scale, float* dx, int64_t rows, int C, void* stream) {
  VLFB_CHECK_ARG(dy && scale && dx && rows >= 0 && C > 0 && (C & 3) == 0);
  const int64_t n4 = rows * (C >> 2);
  if (n4 == 0) return VLFB_OK;
  launch_k(affine_fwd_k, stream_grid(n4, TPB), TPB, 0, ST(stream), (const float4*)dy, (const float4*)scale, nullptr,
                                                             (float4*)dx, n4, C >> 2);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_maxpool3d_fwd(const float* x, float* y, int32_t* argmax, const vlfb_conv_geom_t* g, void* stream) {
  VLFB_CHECK_ARG(x && y && g && (g->C & 3) == 0 && g->Co == g->C);
  const int64_t total = (int64_t)g->N * g->To * g->Ho * g->Wo * (g->C >> 2);
  if (total == 0) return VLFB_OK;
  launch_k(maxpool_fwd_k, stream_grid(total, TPB), TPB, 0, ST(stream), x, y, argmax, *g, total);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_maxpool3d_bwd(const float* dy, const int32_t* argmax, float* dx, const vlfb_conv_geom_t* g, void* stream) {
  VLFB_CHECK_ARG(dy && argmax && dx && g);
  const int64_t total = (int64_t)g->N * g->To * g->Ho * g->Wo * g->C;
  if (total == 0) return VLFB_OK;
  launch_k(maxpool_bwd_k, stream_grid(total, TPB), TPB, 0, ST(stream), dy, argmax, dx, g->C, total);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_maxpool3d_bwd_gather(const float* dy, const int32_t* argmax, const float* y, float* dx,
                               const vlfb_conv_geom_t* g, int tf32_out, void* stream) {
  VLFB_CHECK_ARG(dy && argmax && dx && g && (g->C & 3) == 0 && g->Co == g->C);
  VLFB_CHECK_ARG(g->sT > 0 && g->sH > 0 && g->sW > 0 && (int64_t)g->N * g->T * g->H * g->W < (1ll << 31));
  const int64_t total = (int64_t)g->N * g->T * g->H * g->W * (g->C >> 2);
  if (total == 0) return VLFB_OK;
  launch_k(maxpool_bwd_gather_k, stream_grid(total, TPB), TPB, 0, ST(stream), dy, argmax, y, dx, *g, total, tf32_out);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_avgpool3d_fwd(const float* x, float* y, const vlfb_conv_geom_t* g, void* stream) {
  VLFB_CHECK_ARG(x && y && g && (g->C & 3) == 0 && g->pT == 0 && g->pH == 0 && g->pW == 0);
  const int64_t total = (int64_t)g->N * g->To * g->Ho * g->Wo * (g->C >> 2);
  if (total == 0) return VLFB_OK;
  launch_k(avgpool_fwd_k, stream_grid(total, TPB), TPB, 0, ST(stream), x, y, *g, total);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_avgpool3d_bwd(const float* dy, float* dx, const vlfb_conv_geom_t* g, int accumulate, void* stream) {
  VLFB_CHECK_ARG(dy && dx && g && (g->C & 3) == 0 && g->pT == 0 && g->pH == 0 && g->pW == 0);
  const int64_t total = (int64_t)g->N * g->T * g->H * g->W * (g->C >> 2);
  if (total == 0) return VLFB_OK;
  launch_k(avgpool_bwd_k, stream_grid(total, TPB), TPB, 0, ST(stream), dy, dx, *g, accumulate, total);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_roi_align_fwd(const float* feat, const float* rois, float* out, int N, int H, int W, int C, int R, int PH,
                       int PW, float spatial_scale, int sampling_ratio, void* stream) {
  VLFB_CHECK_ARG(feat && rois && out && N > 0 && H > 0 && W > 0 && (C & 3) == 0 && R >= 0 && PH > 0 && PW > 0);
  const int64_t total = (int64_t)R * PH * PW * (C >> 2);
  if (total == 0) return VLFB_OK;
  launch_k(roi_align_fwd_k, stream_grid(total, TPB), TPB, 0, ST(stream), feat, rois, out, H, W, C, PH, PW, spatial_scale,
                                                                  sampling_ratio, total);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_roi_align_bwd(const float* dout, const float* rois, float* dfeat, int N, int H, int W, int C, int R, int PH,
                       int PW, float spatial_scale, int sampling_ratio, void* stream) {
  VLFB_CHECK_ARG(dout && rois && dfeat && N > 0 && H > 0 && W > 0 && (C & 3) == 0 && R >= 0 && PH > 0 && PW > 0 &&
                 PW <= ROI_BWD_MAX_PW);
  const int64_t total = (int64_t)N * H * W * (C >> 2);
  if (R == 0) return VLFB_OK;
  launch_k(roi_align_bwd_k, stream_grid(total, TPB), TPB, 0, ST(stream), dout, rois, dfeat, H, W, C, R, PH, PW,
           spatial_scale, sampling_ratio, total);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_roi_align_table(const float* rois, int32_t* pos, float* w, int32_t* grid, int H, int W, int R, int PH, int PW,
                         int max_grid, float spatial_scale, int sampling_ratio, void* stream) {
  VLFB_CHECK_ARG(rois && pos && w && grid && R >= 0 && max_grid > 0);
  const int64_t total = (int64_t)R * PH * PW * max_grid * max_grid;
  if (total == 0) return VLFB_OK;
  launch_k(roi_table_k, stream_grid(total, TPB), TPB, 0, ST(stream), rois, pos, w, grid, H, W, R, PH, PW, max_grid,
                                                              spatial_scale, sampling_ratio);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_softmax_fwd(const float* x, float* p, int64_t rows, int cols, float scale, int tf32, void* stream) {
  VLFB_CHECK_ARG(x && p && rows >= 0 && cols > 0);
  if (rows == 0) return VLFB_OK;
  launch_k(softmax_fwd_k, stream_grid(rows, TPB / 32), TPB, 0, ST(stream), x, p, rows, cols, scale, tf32);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_softmax_bwd(const float* p, const float* dp, float* dx, int64_t rows, int cols, float scale, int tf32, void* stream) {
  VLFB_CHECK_ARG(p && dp && dx && rows >= 0 && cols > 0);
  if (rows == 0) return VLFB_OK;
  launch_k(softmax_bwd_k, stream_grid(rows, TPB / 32), TPB, 0, ST(stream), p, dp, dx, rows, cols, scale, tf32);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_layernorm_fwd(const float* x, float* y, float* mean, float* std, int64_t rows, int cols, float eps,
                       void* stream) {
  VLFB_CHECK_ARG(x && y && rows >= 0 && cols > 0);
  if (rows == 0) return VLFB_OK;
  launch_k(layernorm_fwd_k, stream_grid(rows, TPB / 32), TPB, 0, ST(stream), x, y, mean, std, rows, cols, eps);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_layernorm_bwd(const float* dy, const float* y, const float* std, float* dx, int64_t rows, int cols,
                       void* stream) {
  VLFB_CHECK_ARG(dy && y && std && dx && rows >= 0 && cols > 0);
  if (rows == 0) return VLFB_OK;
  launch_k(layernorm_bwd_k, stream_grid(rows, TPB / 32), TPB, 0, ST(stream), dy, y, std, dx, rows, cols);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_relu_fwd(const float* x, float* y, int64_t n, void* stream) {
  VLFB_CHECK_ARG(x && y && n >= 0);
  return ew_launch<EW_RELU>(x, nullptr, y, n, 0.f, 0.f, ST(stream));
}
int vlfb_relu_bwd(const float* dy, const float* y, float* dx, int64_t n, void* stream) {
  VLFB_CHECK_ARG(dy && y && dx && n >= 0);
  return ew_launch<EW_RELU_BWD>(dy, y, dx, n, 0.f, 0.f, ST(stream));
}
int vlfb_axpby(const float* x, float a, const float* y, float b, float* out, int64_t n, void* stream) {
  VLFB_CHECK_ARG(x && out && n >= 0 && (y || b == 0.f));
  return ew_launch<EW_AXPBY>(x, y, out, n, a, b, ST(stream));
}
int vlfb_fill(float* x, float v, int64_t n, void* stream) {
  VLFB_CHECK_ARG(x && n >= 0);
  return ew_launch<EW_FILL>(nullptr, nullptr, x, n, v, 0.f, ST(stream));
}
int vlfb_round_tf32(const float* x, float* y, int64_t n, void* stream) {
  VLFB_CHECK_ARG(x && y && n >= 0);
  return ew_launch<EW_TF32>(x, nullptr, y, n, 0.f, 0.f, ST(stream));
}
int vlfb_add_tf32(const float* x, const float* y, float* out, int64_t n, void* stream) {
  VLFB_CHECK_ARG(x && y && out && n >= 0);
  return ew_launch<EW_ADD_TF32>(x, y, out, n, 0.f, 0.f, ST(stream));
}
int vlfb_relu_tf32(const float* x, float* y, int64_t n, void* stream) {
  VLFB_CHECK_ARG(x && y && n >= 0);
  return ew_launch<EW_RELU_TF32>(x, nullptr, y, n, 0.f, 0.f, ST(stream));
}
int vlfb_relu_bits(const float* x, uint32_t* bits, int64_t n, void* stream) {
  VLFB_CHECK_ARG(x && bits && n >= 0 && (n & 31) == 0);
  return relu_bits(x, bits, n, ST(stream));
}
int vlfb_relu_bwd_tf32(const float* dy, const float* y, float* dx, int64_t n, void* stream) {
  VLFB_CHECK_ARG(dy && y && dx && n >= 0);
  return ew_launch<EW_RELU_BWD_TF32>(dy, y, dx, n, 0.f, 0.f, ST(stream));
}
int vlfb_add_relu_bwd_tf32(const float* a, const float* b, const float* y, float* out, int64_t n, void* stream) {
  VLFB_CHECK_ARG(a && b && out && n >= 0);
  if (n == 0) return VLFB_OK;
  const bool vec = ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(y) |
                     reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  launch_k(add_mask_tf32_k, stream_grid(n, TPB, 4), TPB, 0, ST(stream), a, b, y, out, n, vec ? 1 : 0);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}
// Row slabs of colsum: ~2 waves of 32-column blocks on 148 SMs, at least 64 rows per slab.
static int colsum_slabs(int64_t rows, int cols) {
  const int cb = ceil_div(cols, 32);
  int64_t slabs = (2 * 148 + cb - 1) / cb;
  const int64_t max_slabs = (rows + 63) / 64;
  if (slabs > max_slabs) slabs = max_slabs;
  return slabs < 1 ? 1 : (int)slabs;
}

size_t vlfb_colsum_workspace_bytes(int64_t rows, int cols) {
  if (rows <= 0 || cols <= 0) return 0;
  const int slabs = colsum_slabs(rows, cols);
  return slabs > 1 ? (size_t)slabs * cols * sizeof(float) : 0;
}

int vlfb_colsum(const float* x, int64_t ld, float* out, int64_t rows, int cols, int accumulate, void* workspace,
                size_t workspace_bytes, void* stream) {
  VLFB_CHECK_ARG(x && out && rows >= 0 && cols > 0);
  if (rows == 0) {
    if (accumulate) return VLFB_OK;
    return ew_launch<EW_FILL>(nullptr, nullptr, out, cols, 0.f, 0.f, ST(stream));
  }
  const int slabs = colsum_slabs(rows, cols);
  float* part = nullptr;
  if (slabs > 1) {
    if (!workspace || workspace_bytes < vlfb_colsum_workspace_bytes(rows, cols)) {
      ::vlfb::set_error("vlfb_colsum: workspace of %zu bytes < vlfb_colsum_workspace_bytes() = %zu", workspace_bytes,
                        vlfb_colsum_workspace_bytes(rows, cols));
      return VLFB_E_WORKSPACE;
    }
    part = static_cast<float*>(workspace);
  }
  const int64_t rpb = (rows + slabs - 1) / slabs;
  launch_k(colsum_k, dim3(ceil_div(cols, 32), slabs), dim3(32, 8), 0, ST(stream), x, ld, out, rows, cols, rpb, part,
           accumulate);
  VLFB_CHECK_LAUNCH();
  if (part) {
    launch_k(colsum_finish_k, dim3(ceil_div(cols, TPB)), dim3(TPB), 0, ST(stream), (const float*)part, slabs, out, cols,
             accumulate);
    VLFB_CHECK_LAUNCH();
  }
  return VLFB_OK;
}

int vlfb_sigmoid_fwd(const float* x, float* y, int64_t n, void* stream) {
  VLFB_CHECK_ARG(x && y && n >= 0);
  return ew_launch<EW_SIGMOID>(x, nullptr, y, n, 0.f, 0.f, ST(stream));
}

int vlfb_dropout_fwd(const float* x, float* y, int64_t n, float ratio, uint64_t seed, uint64_t offset,
                     const int64_t* step, void* stream) {
  VLFB_CHECK_ARG(x && y && n >= 0 && ratio >= 0.f && ratio < 1.f);
  if (n == 0) return VLFB_OK;
  launch_k(dropout_k, stream_grid((n + 3) / 4, TPB), TPB, 0, ST(stream), x, y, n, ratio, 1.f / (1.f - ratio), seed, offset,
                                                                   step);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_copy2d(const float* src, int64_t lds, float* dst, int64_t ldd, int64_t rows, int cols, int accumulate,
                void* stream) {
  VLFB_CHECK_ARG(src && dst && rows >= 0 && cols >= 0);
  if (rows * cols == 0) return VLFB_OK;
  launch_k(copy2d_k, stream_grid(rows * cols, TPB), TPB, 0, ST(stream), src, lds, dst, ldd, rows, cols, accumulate);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_nc_to_cl_round(const float* src, float* dst, int N, int C, int64_t inner, int Cpad, int tf32_out, void* stream) {
  VLFB_CHECK_ARG(src && dst && N > 0 && C > 0 && inner > 0 && Cpad >= C);
  if (Cpad == 4 && (inner & 3) == 0 && ((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 15) == 0) {
    const int64_t total = (int64_t)N * (inner >> 2);
    launch_k(nc_to_cl4_k, stream_grid(total, TPB), TPB, 0, ST(stream), src, (float4*)dst, C, inner >> 2, total, tf32_out);
    VLFB_CHECK_LAUNCH();
    return VLFB_OK;
  }
  dim3 grid(ceil_div(inner, 32), ceil_div(Cpad, 32), N), block(32, 8);
  launch_k(nc_to_cl_k, grid, block, 0, ST(stream), src, dst, C, inner, Cpad, tf32_out);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_nc_to_cl_pitched(const float* src, float* dst, int N, int C, int64_t inner, int Cpad, int tf32_out, int W, int pitch,
                          int left, void* stream) {
  VLFB_CHECK_ARG(src && dst && N > 0 && C > 0 && C <= 4 && Cpad == 4 && inner > 0 && W > 0 && (W & 3) == 0);
  VLFB_CHECK_ARG(inner % W == 0 && left >= 0 && pitch >= left + W);
  VLFB_CHECK_ARG(((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 15) == 0);
  const int64_t total = (int64_t)N * (inner >> 2);
  launch_k(nc_to_cl4p_k, stream_grid(total, TPB), TPB, 0, ST(stream), src, (float4*)dst, C, inner >> 2, total, tf32_out, W >> 2,
           pitch, left);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_nc_to_cl(const float* src, float* dst, int N, int C, int64_t inner, int Cpad, void* stream) {
  return vlfb_nc_to_cl_round(src, dst, N, C, inner, Cpad, 0, stream);
}

int vlfb_cl_to_nc(const float* src, float* dst, int N, int C, int64_t inner, int Cpad, void* stream) {
  VLFB_CHECK_ARG(src && dst && N > 0 && C > 0 && inner > 0 && Cpad >= C);
  dim3 grid(ceil_div(inner, 32), ceil_div(C, 32), N), block(32, 8);
  launch_k(cl_to_nc_k, grid, block, 0, ST(stream), src, dst, C, inner, Cpad);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_weight_transpose(const float* w, float* wt, const float* scale, int Co, int taps, int Ci, void* stream) {
  VLFB_CHECK_ARG(w && wt && Co > 0 && taps > 0 && Ci > 0);
  dim3 grid(ceil_div(Ci, 32), ceil_div(Co, 32), taps), block(32, 8);
  launch_k(weight_transpose_k, grid, block, 0, ST(stream), w, wt, scale, Co, taps, Ci);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_weight_transpose_multi(const vlfb_wt_job_t* jobs, int njobs, int total_blocks, void* stream) {
  VLFB_CHECK_ARG(jobs && njobs > 0 && total_blocks > 0);
  launch_k(weight_transpose_multi_k, dim3(total_blocks), dim3(32, 8), 0, ST(stream), jobs, njobs);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_sigmoid_ce_fwd(const float* logits, const int32_t* targets, float* loss, int64_t n, float scale, void* stream) {
  VLFB_CHECK_ARG(logits && targets && loss && n > 0);
  launch_k(sigmoid_ce_fwd_k, 1, 1024, 0, ST(stream), logits, targets, loss, n, scale);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_sigmoid_ce_bwd(const float* logits, const int32_t* targets, const float* dloss, float* dlogits, int64_t n,
                        float scale, void* stream) {
  VLFB_CHECK_ARG(logits && targets && dlogits && n > 0);
  launch_k(sigmoid_ce_bwd_k, 1, 1024, 0, ST(stream), logits, targets, dloss, dlogits, n, scale);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_softmax_ce_fwd(const float* logits, const int32_t* labels, float* prob, float* loss, int rows, int cols,
                        float scale, void* stream) {
  VLFB_CHECK_ARG(logits && labels && prob && loss && rows > 0 && cols > 0);
  launch_k(softmax_ce_fwd_k, 1, 256, 0, ST(stream), logits, labels, prob, loss, rows, cols, scale);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_softmax_ce_bwd(const float* prob, const int32_t* labels, float* dlogits, int rows, int cols, float scale,
                        void* stream) {
  VLFB_CHECK_ARG(prob && labels && dlogits && rows > 0 && cols > 0);
  launch_k(softmax_ce_bwd_k, stream_grid((int64_t)rows * cols, TPB), TPB, 0, ST(stream), prob, labels, dlogits, rows, cols,
                                                                                  scale);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

int vlfb_sgd_nesterov(float* p, float* g, float* m, float* p_tf32, int64_t n, const float* lr, float momentum, float wd,
                      int nesterov, void* stream) {
  VLFB_CHECK_ARG(p && g && m && lr && n >= 0);
  if (n == 0) return VLFB_OK;
  launch_k(sgd_k, stream_grid(n, TPB, 4), TPB, 0, ST(stream), p, g, m, p_tf32, n, lr, momentum, wd, nesterov);
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

}  // extern "C"
