/*
 * vlfb.h -- C ABI of libvlfb.so: the B200 (sm_100a) hot path of
 * facebookresearch/video-long-term-feature-banks (R50/R101-I3D-NL backbone fwd/bwd +
 * Feature-Bank-Operator attention).
 *
 * The reference has no FFI of its own: its hot path sits behind the Caffe2 operator
 * registry (REGISTER_CUDA_OPERATOR, caffe2_customized_ops/video/affine_nd_op.cu:106-109)
 * and the CNNModelHelper op emitters called from lib/models/*.py.  Each entry point
 * below names the reference operator call site(s) it replaces (file:line relative to
 * the reference root).  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless named host_*; the caller owns all memory
 *   - activations are fp32, channels-last ("NDHWC": [N][T][H][W][C]); conv weights are
 *     [Cout][kT][kH][kW][Cin]
 *   - all calls are asynchronous on `stream` (a cudaStream_t passed as void*), never
 *     synchronise, never allocate, keep no mutable global state (engine / tiling choices are per-call
 *     fields of vlfb_gemm_params_t; the only process state is immutable: cached driver entry points,
 *     occupancy queries and environment overrides read once)
 *   - return value: 0 = ok, <0 = error (see VLFB_E_*); vlfb_last_error() gives the text
 */
#ifndef VLFB_H_
#define VLFB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VLFB_OK 0
#define VLFB_E_BADARG (-1)
#define VLFB_E_UNSUPPORTED (-2)
#define VLFB_E_CUDA (-3)
#define VLFB_E_WORKSPACE (-4)   /* caller-provided workspace too small (see the *_workspace query) */

/* Storage types of operands that are not fp32 (fp32 is the parity mode of every other entry point). */
typedef enum { VLFB_DT_F32 = 0, VLFB_DT_BF16 = 1 } vlfb_dtype_t;

/* ---- library ------------------------------------------------------------------------- */
int vlfb_version(void);                 /* 100 * major + minor */
const char* vlfb_last_error(void);      /* thread-local message of the last failing call */

/* ---- gathered GEMM: D[m,n] = epi( sum_k A[m,k] * B[n,k] ) ------------------------------ */
/* One descriptor per operand.  `kind`:
 *   VLFB_OP_DENSE_K   rows (m or n) at ptr + batch*batch_stride + row*ld, k contiguous
 *   VLFB_OP_DENSE_MN  rows indexed by k at ptr + batch*batch_stride + k*ld, m (or n) contiguous
 *   VLFB_OP_CONV_K    A of conv forward : row m = output position, k = (tap, cin)
 *   VLFB_OP_DGRAD_K   A of conv dgrad   : row m = input position,  k = (tap, cout)
 *   VLFB_OP_CONV_MN   B of conv wgrad   : k = output position, n = (kh,kw,cin), one kt per z-slice
 *   VLFB_OP_STEM_K / VLFB_OP_STEM_MN    conv1 (Cin padded to 4): k (resp. n) = (kt,kh) x (8 pixels x 4 ch).
 *                     ptr = first real pixel; ld = row pitch in PIXELS (0 = W).  With zero pad pixels around every row
 *                     (pW to the left, pitch >= max(pW + W, (Wo-1)*sW + 8)) and Wo % 16 == 0 the operand is staged by TMA
 *                     (overlapping-window tensor map) instead of 16-byte cp.async gathers.
 */
enum {
  VLFB_OP_DENSE_K = 0, VLFB_OP_DENSE_MN = 1, VLFB_OP_CONV_K = 2, VLFB_OP_DGRAD_K = 3,
  VLFB_OP_CONV_MN = 4, VLFB_OP_STEM_K = 5, VLFB_OP_STEM_MN = 6
};

typedef struct {
  int N, T, H, W, C;          /* input tensor  [N][T][H][W][C]              */
  int To, Ho, Wo, Co;         /* output tensor [N][To][Ho][Wo][Co]          */
  int kT, kH, kW;             /* filter taps                                 */
  int sT, sH, sW;             /* strides                                     */
  int pT, pH, pW;             /* symmetric zero padding                      */
  int dT, dH, dW;             /* dilations                                   */
} vlfb_conv_geom_t;

typedef struct {
  const float* ptr;
  int kind;                   /* VLFB_OP_*                                   */
  int64_t ld;                 /* DENSE_*: elements between consecutive rows  */
  int64_t batch_stride;       /* DENSE_*: elements between batches           */
} vlfb_operand_t;

/* VLFB_EPI_TF32: round the stored value to TF32 (round-to-nearest, ties away: cvt.rna.tf32.f32) so that a
 * consumer GEMM reads operands that the tensor core would otherwise truncate. */
/* VLFB_EPI_ACCUM: the previous contents of d are added like a residual (v += d, then ReLU / mask / rounding). */
enum { VLFB_EPI_RELU = 1, VLFB_EPI_ACCUM = 2, VLFB_EPI_ATOMIC = 4, VLFB_EPI_TF32 = 8 };

typedef struct {
  vlfb_operand_t a, b;
  vlfb_conv_geom_t g;         /* used by the CONV_ / DGRAD_ / STEM_ kinds    */
  int M, N, K;                /* logical GEMM extent (K per z-slice for wgrad) */
  int batch;                  /* >= 1 (DENSE only)                           */
  int taps;                   /* wgrad: number of temporal taps kT (z-slices), else 1 */
  int split_k;                /* >= 1 (>1 needs VLFB_EPI_ATOMIC); 0 = the library picks it with the tile width.  With
                               * VLFB_EPI_ATOMIC, split_k == 0 and a workspace (stream_k >= 0) the product is never
                               * split into K slices that add into d in arrival order: it runs as whole tiles or as
                               * stream-K pieces summed in a fixed order, so the result is the same in every run.
                               * Without a workspace, or with stream_k == -1, the library may pick plain split-K,
                               * whose atomic additions make the last bits depend on the order the slices finish. */
  float* d;                   /* output rows: d + batch*d_batch_stride + m*ldd + n (+ tap*d_tap_stride) */
  int64_t ldd, d_batch_stride, d_tap_stride;
  float alpha;                /* applied first                               */
  const float* col_scale;     /* [N] or NULL : v = v*col_scale[n]            */
  const float* col_bias;      /* [N] or NULL : v += col_bias[n]              */
  const float* row_scale;     /* [M] or NULL : v *= row_scale[m]             */
  const float* residual;      /* same addressing as d, or NULL : v += res    */
  const float* relu_mask;     /* same addressing as d, or NULL : v = mask > 0 ? v : 0  (applied after the
                               * residual / ReLU, before the TF32 rounding).  Backward of a ReLU fused into the
                               * dgrad GEMM that produces the gradient: mask = the ReLU's output */
  int flags;                  /* VLFB_EPI_*                                  */
  /* ---- per-call execution options (0 = library default) ---- */
  void* workspace;            /* stream-K scratch (partial tiles + arrival counters) of >= vlfb_gemm_workspace_bytes()
                               * bytes, 16-byte aligned, ZERO-FILLED ONCE by the caller before its first use and then
                               * only touched by vlfb_gemm (the counters are zero again when a launch ends); calls that
                               * share it must be ordered on one stream.  NULL: no stream-K fix-ups (see split_k). */
  size_t workspace_bytes;
  int engine;                 /* VLFB_ENGINE_TCGEN05 (0, default) or VLFB_ENGINE_SIMT (fp32 cross-check engine) */
  int tile_n;                 /* 0 = chosen by the library, else the output-tile width (32..256, multiple of 32) */
  int pair;                   /* 0 = auto, 1 = CTA pairs (cta_group::2, 256-row tiles) whenever legal, -1 = never */
  int stream_k;               /* 0 = auto, 1 = stream-K whenever legal, -1 = never */
  /* ---- ReLU sign bits: one bit per element of d (bit e & 31 of word e >> 5, e = the element's offset from d) ---- */
  const uint32_t* relu_mask_bits; /* or NULL: v = bit ? v : 0, applied where relu_mask is (not both).  The mask of a ReLU's
                               * backward at 1/32 of the bytes of the activation itself. */
  uint32_t* relu_bits_out;    /* or NULL: with VLFB_EPI_RELU, bit = (stored value > 0).  Dense outputs only: ldd == N,
                               * N % 32 == 0, batch == taps == split_k == 1, no VLFB_EPI_ATOMIC; M * N / 32 words. */
} vlfb_gemm_params_t;

enum { VLFB_ENGINE_TCGEN05 = 0, VLFB_ENGINE_SIMT = 1 };

/* What vlfb_gemm would do for `p` (host-only, no launch). */
typedef struct {
  int tile_n;                 /* output-tile width */
  int split_k;                /* plain split-K factor (atomic epilogues) */
  int pair;                   /* 1: 256 x tile_n tiles on CTA pairs (tcgen05 cta_group::2) */
  int stream_k;               /* 1: equal (tile, K-chunk) ranges per SM (pair), shared tiles fixed up in the workspace */
  int tiles;                  /* output tiles (x split_k) */
  int units;                  /* CTAs (or CTA pairs) of the persistent grid */
} vlfb_gemm_plan_t;

/* Replaces: Caffe2 Conv (cuDNN) at resnet_video.py:169-179, model_builder_video.py:211-217,
 * nonlocal_helper.py:36-78,131-144, lfb_helper.py:175-202,244-251,305-334; its gradients;
 * BatchMatMul (cuBLAS) at nonlocal_helper.py:94-95,121 and lfb_helper.py:223-224,234;
 * FC at resnet_video.py:327-331; and the AffineNd / Relu / Sum epilogues that follow
 * them (model_builder_video.py:218-219, resnet_helper.py:112-117). */
int vlfb_gemm(const vlfb_gemm_params_t* p, void* stream);
/* Host-only query: the tiling / schedule vlfb_gemm would use for `p` on a device with `num_sms` SMs (<= 0: 148),
 * assuming every operand is TMA-addressable.  No launch, no device access. */
int vlfb_gemm_plan(const vlfb_gemm_params_t* p, int num_sms, vlfb_gemm_plan_t* plan);
/* Bytes of vlfb_gemm_params_t.workspace that enable stream-K for every problem size (a constant of the build). */
size_t vlfb_gemm_workspace_bytes(void);

/* ---- AffineNd (standalone; caffe2_customized_ops/video/affine_nd_op.cu:62-104) ---------- */
int vlfb_affine_nd_fwd(const float* x, const float* scale, const float* bias, float* y,
                       int64_t rows, int C, void* stream);
int vlfb_affine_nd_bwd(const float* dy, const float* scale, float* dx, int64_t rows, int C,
                       void* stream);

/* ---- SpatialBN (trainable batch normalisation; replaces Caffe2 SpatialBN / SpatialBNGradient as emitted by
 *      model_builder_video.py:176-197 Conv3dBN, resnet_video.py:185-188, nonlocal_helper.py:146-155).
 *      x, y, dy, dx: channels-last [rows][C] (rows = N*T*H*W), C % 4 == 0.  Per-channel vectors are C floats.
 *      `workspace` (>= vlfb_spatial_bn_workspace_bytes(C), 16-byte aligned, owned by the caller) holds the fp64
 *      reduction accumulators and the per-channel coefficients of the apply pass between the call's launches.
 *   fwd   (is_test = False): batch mean / biased variance over the rows -> saved_mean (`_bn_sm`), saved_inv_std
 *         = 1/sqrt(var + eps) (`_bn_siv`, read by lib/utils/bn_helper.py:170-173); y = (x - mean) * inv_std * scale
 *         + bias; running_mean (`_bn_rm`) = running_mean * momentum + mean * (1 - momentum), running_var (`_bn_riv`:
 *         a VARIANCE despite its name, bn_helper.py:216-219) likewise from the unbiased batch variance; both may be
 *         NULL (bn_aux_model of precise-BN ignores them).
 *   infer (is_test = True): y = (x - running_mean) / sqrt(running_var + eps) * scale + bias.
 *   bwd:  dx; dscale += sum dy * xhat, dbias += sum dy (either may be NULL).                                        */
size_t vlfb_spatial_bn_workspace_bytes(int C);
int vlfb_spatial_bn_fwd(const float* x, const float* scale, const float* bias, float* running_mean, float* running_var,
                        float* saved_mean, float* saved_inv_std, float* y, int64_t rows, int C, float eps, float momentum,
                        void* workspace, size_t workspace_bytes, void* stream);
int vlfb_spatial_bn_infer(const float* x, const float* scale, const float* bias, const float* running_mean,
                          const float* running_var, float* y, int64_t rows, int C, float eps, void* workspace,
                          size_t workspace_bytes, void* stream);
int vlfb_spatial_bn_bwd(const float* dy, const float* x, const float* scale, const float* saved_mean,
                        const float* saved_inv_std, float* dx, float* dscale, float* dbias, int64_t rows, int C,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- pooling (MaxPool/AveragePool: resnet_video.py:190-196,219-225, nonlocal_helper.py:48-54,
 *      head_helper.py:37-40,92-98,113-115) -------------------------------------------------- */
int vlfb_maxpool3d_fwd(const float* x, float* y, int32_t* argmax /* may be NULL */,
                       const vlfb_conv_geom_t* g, void* stream);
int vlfb_maxpool3d_bwd(const float* dy, const int32_t* argmax, float* dx /* pre-zeroed or accumulated */,
                       const vlfb_conv_geom_t* g, void* stream);
/* Gather form of the max-pool backward: dx (written completely, no pre-zeroing, no atomics) = for every input element the
 * sum of dy over the windows that cover it and whose argmax it is.  y (may be NULL) = the pool's forward OUTPUT: windows
 * whose maximum is <= 0 pass no gradient, i.e. the backward of a ReLU that produced the pool's input is folded in
 * (resnet_video.py:189-196: conv1 -> AffineNd -> Relu -> MaxPool 'pool1'); tf32_out rounds dx (a GEMM operand). */
int vlfb_maxpool3d_bwd_gather(const float* dy, const int32_t* argmax, const float* y, float* dx,
                              const vlfb_conv_geom_t* g, int tf32_out, void* stream);
int vlfb_avgpool3d_fwd(const float* x, float* y, const vlfb_conv_geom_t* g, void* stream);
int vlfb_avgpool3d_bwd(const float* dy, float* dx, const vlfb_conv_geom_t* g, int accumulate,
                       void* stream);

/* ---- RoIAlign, legacy Caffe2 semantics (lfb_helper.py:130-152) ------------------------ */
/* feat [N][H][W][C], rois [R][5] = (batch, x1, y1, x2, y2), out [R][PH][PW][C] */
int vlfb_roi_align_fwd(const float* feat, const float* rois, float* out, int N, int H, int W,
                       int C, int R, int PH, int PW, float spatial_scale, int sampling_ratio,
                       void* stream);
/* Backward in gather form: each element of dfeat adds the contributions of every RoI bin in a fixed order (same result
 * in every run); PW <= 32. */
int vlfb_roi_align_bwd(const float* dout, const float* rois, float* dfeat /* accumulated */,
                       int N, int H, int W, int C, int R, int PH, int PW, float spatial_scale,
                       int sampling_ratio, void* stream);
/* Bilinear sample table for bit-exact index tests: per (r,ph,pw,iy,ix) with iy,ix < max_grid:
 * pos[4] (y*W+x or -1) and w[4]; grid[r][2] = (grid_h, grid_w). */
int vlfb_roi_align_table(const float* rois, int32_t* pos, float* w, int32_t* grid, int H, int W,
                         int R, int PH, int PW, int max_grid, float spatial_scale,
                         int sampling_ratio, void* stream);

/* ---- row softmax with fused pre-scale (Scale+Softmax: nonlocal_helper.py:96-105,
 *      lfb_helper.py:226-231) -------------------------------------------------------------- */
/* tf32 != 0: store TF32-rounded probabilities (they are the A operand of the next GEMM) */
int vlfb_softmax_fwd(const float* x, float* p, int64_t rows, int cols, float scale, int tf32, void* stream);
/* tf32 != 0: store the TF32-rounded gradient (when it is the only contribution to a GEMM operand) */
int vlfb_softmax_bwd(const float* p, const float* dp, float* dx, int64_t rows, int cols, float scale, int tf32,
                     void* stream);

/* ---- LayerNorm(axis=1, eps, no affine) over rows (lfb_helper.py:160-167,253-256) ------- */
int vlfb_layernorm_fwd(const float* x, float* y, float* mean, float* std, int64_t rows, int cols,
                       float eps, void* stream);
int vlfb_layernorm_bwd(const float* dy, const float* y, const float* std, float* dx, int64_t rows,
                       int cols, void* stream);

/* ---- elementwise ------------------------------------------------------------------------ */
int vlfb_relu_fwd(const float* x, float* y, int64_t n, void* stream);
int vlfb_relu_bwd(const float* dy, const float* y, float* dx, int64_t n, void* stream); /* dx = dy*(y>0) */
int vlfb_axpby(const float* x, float a, const float* y, float b, float* out, int64_t n, void* stream);
int vlfb_fill(float* x, float v, int64_t n, void* stream);
/* TF32-rounding variants used where the result feeds a tensor-core GEMM */
int vlfb_add_tf32(const float* x, const float* y, float* out, int64_t n, void* stream);   /* round(x+y) */
int vlfb_relu_tf32(const float* x, float* y, int64_t n, void* stream);                    /* round(max(x,0)) */
/* bits[e >> 5] bit (e & 31) = x[e] > 0 for e < n (n % 32 == 0): the mask vlfb_gemm_params_t.relu_mask_bits reads,
 * for activations that were not produced by a vlfb_gemm with relu_bits_out. */
int vlfb_relu_bits(const float* x, uint32_t* bits, int64_t n, void* stream);
int vlfb_relu_bwd_tf32(const float* dy, const float* y, float* dx, int64_t n, void* stream); /* round(dy*(y>0)) */
/* out = (y == NULL || y > 0) ? round_tf32(a + b) : 0 : sum of two gradient contributions + ReLU backward + TF32
 * rounding in one pass (out may alias a or b). */
int vlfb_add_relu_bwd_tf32(const float* a, const float* b, const float* y, float* out, int64_t n, void* stream);
/* out[c] (+)= sum_r x[r*ld + c]  (bias gradients of Conv/FC).  Slabs of rows are summed by separate CTAs and their
 * partial sums added in slab order through `workspace` (>= vlfb_colsum_workspace_bytes(rows, cols) bytes, owned by
 * the caller; 0 bytes: one slab), so the result is the same in every run.  Calls that share a workspace must be
 * ordered on one stream. */
size_t vlfb_colsum_workspace_bytes(int64_t rows, int cols);
int vlfb_colsum(const float* x, int64_t ld, float* out, int64_t rows, int cols, int accumulate, void* workspace,
                size_t workspace_bytes, void* stream);
/* y = round-to-nearest TF32 of x (operand preparation for kind::tf32 MMAs; y may alias x) */
int vlfb_round_tf32(const float* x, float* y, int64_t n, void* stream);
int vlfb_sigmoid_fwd(const float* x, float* y, int64_t n, void* stream);
/* Dropout (Caffe2 train mode: y = x*mask/(1-ratio)); mask = Philox(seed, counter) >= ratio with
 * counter = offset + i/4 + (step ? step[0] << 32 : 0).  `step` is an optional DEVICE scalar so that a
 * captured CUDA graph draws a fresh mask at every replay.  The same call on dy is the backward. */
int vlfb_dropout_fwd(const float* x, float* y, int64_t n, float ratio, uint64_t seed, uint64_t offset,
                     const int64_t* step, void* stream);
/* 2-D strided copy: dst[r*ldd + c] = src[r*lds + c] (Concat / slicing; head_helper.py:82-85) */
int vlfb_copy2d(const float* src, int64_t lds, float* dst, int64_t ldd, int64_t rows, int cols,
                int accumulate, void* stream);
/* layout: NCTHW (reference blob layout) <-> NDHWC; inner = T*H*W */
int vlfb_nc_to_cl(const float* src, float* dst, int N, int C, int64_t inner, int Cpad, void* stream);
/* the same with the TF32 rounding of the result fused (tf32_out != 0): the dequeue of a fed clip (`data` blob,
 * model_builder_video.py:335-345) is ONE pass: NCTHW fp32 -> NDHWC, C 3 -> 4, rounded conv1 operand */
int vlfb_nc_to_cl_round(const float* src, float* dst, int N, int C, int64_t inner, int Cpad, int tf32_out, void* stream);
/* the same into W-padded rows: inner = rows * W; row r's W real pixels go to dst pixels [r*pitch + left, +W); the pad
 * pixels are not written (the caller zero-fills the buffer once).  C <= 4 = Cpad, W % 4 == 0.  The stem (conv1) operand. */
int vlfb_nc_to_cl_pitched(const float* src, float* dst, int N, int C, int64_t inner, int Cpad, int tf32_out, int W, int pitch,
                          int left, void* stream);
int vlfb_cl_to_nc(const float* src, float* dst, int N, int C, int64_t inner, int Cpad, void* stream);
/* weights: wt[ci][tap][co] = round_tf32( w[co][tap][ci] * (scale ? scale[co] : 1) )  (dgrad B operand) */
int vlfb_weight_transpose(const float* w, float* wt, const float* scale, int Co, int taps, int Ci,
                          void* stream);
/* All dgrad weight operands of a step in ONE launch (81 convolutions -> 81 tiny kernels otherwise): `jobs` is a
 * device array; job i owns the blocks [block_begin, next block_begin) of ceil(Ci/32) x ceil(Co/32) x taps tiles. */
typedef struct {
  const float* w;             /* [Co][taps][Ci] master weights                */
  float* wt;                  /* [Ci][taps][Co] = round_tf32(w * scale[co])    */
  const float* scale;         /* [Co] or NULL                                 */
  int Co, taps, Ci;
  int block_begin;
} vlfb_wt_job_t;
int vlfb_weight_transpose_multi(const vlfb_wt_job_t* jobs, int njobs, int total_blocks, void* stream);

/* ---- losses (resnet_video.py:333-349) --------------------------------------------------- */
/* Detectron SigmoidCrossEntropyLoss: loss[0] = scale * sum(per-elt) / max(#valid,1e-5) */
int vlfb_sigmoid_ce_fwd(const float* logits, const int32_t* targets, float* loss, int64_t n,
                        float scale, void* stream);
int vlfb_sigmoid_ce_bwd(const float* logits, const int32_t* targets, const float* dloss /* device scalar or NULL=1 */,
                        float* dlogits, int64_t n, float scale, void* stream);
int vlfb_softmax_ce_fwd(const float* logits, const int32_t* labels, float* prob, float* loss,
                        int rows, int cols, float scale, void* stream);
int vlfb_softmax_ce_bwd(const float* prob, const int32_t* labels, float* dlogits, int rows, int cols,
                        float scale, void* stream);

/* ---- optimizer: WeightedSum + MomentumSGDUpdate fused (model_builder_video.py:375-388) -- */
/* p_tf32 (may be NULL): also writes the TF32-rounded copy of the updated parameter (GEMM operand). */
int vlfb_sgd_nesterov(float* p, float* g, float* m, float* p_tf32, int64_t n,
                      const float* lr /* device scalar */, float momentum, float wd, int nesterov,
                      void* stream);

/* ---- inference-mode FBO-NL over the RAW bank (csrc/fbo.cu) --------------------------------
 * Replaces, per FBO-NL layer of a test-mode graph (no dropout between 'lfb_1x1' and phi/g), the operators
 * Conv 'lfb_1x1' (lfb_helper.py:320-338), Conv '{prefix}_phi' / '{prefix}_g' (:183-202), BatchMatMul / Scale /
 * Softmax / BatchMatMul (:223-234) by ONE pass over the bank: with q = W_1^T W_phi^T theta (computed by the caller),
 *   out[r][:] = sum_j softmax_j(scale * q[r].bank[r][j]) * bank[r][j][:]            (then y = W_g (W_1 out + c_1) + c_g).
 * bank [R][L][D] fp32 (D in {1024, 2048, 4096}), q [R][D], out [R][D]; prob [R][L] optional (NULL: not kept).
 * tf32_out != 0 rounds `out` to TF32 (it feeds a tensor-core matmul).  The L rows of a RoI are split over
 * vlfb_fbo_bank_scan_splits() CTAs whose partial (max, sum, weighted rows) land in `workspace`. */
int vlfb_fbo_bank_scan_splits(int R, int L, int D);
size_t vlfb_fbo_bank_scan_workspace(int R, int L, int D);
int vlfb_fbo_bank_scan(const float* bank, const float* q, float scale, float* out, float* prob, int R, int L, int D,
                       int tf32_out, void* workspace, size_t workspace_bytes, void* stream);
/* The same scan over a bank stored as `bank_dtype` (vlfb_dtype_t): VLFB_DT_F32 (D = 1024 / 2048 / 4096) or
 * VLFB_DT_BF16 (D = 2048 / 4096; half the HBM bytes per row -- BASELINE configs[4] "fp32 and bf16 banks").  Queries,
 * scores, softmax and the weighted sum stay fp32.  The splits / workspace queries depend on the storage type (a tile
 * is 64 KB of rows either way).  vlfb_cast_f32_to_bf16 (round to nearest even, n % 8 == 0) produces such a bank. */
int vlfb_fbo_bank_scan_splits_dt(int R, int L, int D, int bank_dtype);
size_t vlfb_fbo_bank_scan_workspace_dt(int R, int L, int D, int bank_dtype);
int vlfb_fbo_bank_scan_dt(const void* bank, int bank_dtype, const float* q, float scale, float* out, float* prob, int R,
                          int L, int D, int tf32_out, void* workspace, size_t workspace_bytes, void* stream);
int vlfb_cast_f32_to_bf16(const float* x, void* y, int64_t n, void* stream);

/* ---- training-mode FBO-NL stack, one launch per direction (csrc/fbo.cu section 3) ---------------------
 * Replaces, for ALL layers of lfb_helper.NLLayers (:266-292) with one query per RoI and FBO_NL.PRE_ACT, the operators of
 * NLCore (:170-263): Conv theta / phi / g, BatchMatMul, Scale, Softmax, BatchMatMul, LayerNorm, Relu, Conv out, Dropout,
 * Sum -- phi and g are folded onto the shared projected bank bp (prepare_lfb :320-338 output, after its dropout):
 * score_j = (W_phi^T theta) . bp_j (+ const), y = W_g (sum_j p_j bp_j) + b_g.  Weights are [out][in] row-major fp32. */
typedef struct {
  const float *w_theta, *b_theta;   /* [d][dA], [d] or NULL   '{prefix}_theta_w/_b'  */
  const float *w_phi, *b_phi;       /* [d][dB], [d] or NULL   '{prefix}_phi_w/_b'    */
  const float *w_g, *b_g;           /* [d][dB], [d] or NULL   '{prefix}_g_w/_b'      */
  const float *w_out, *b_out;       /* [dA][d], [dA] or NULL  '{prefix}_out_w/_b'    */
  float *gw_theta, *gb_theta, *gw_phi, *gb_phi, *gw_g, *gb_g, *gw_out, *gb_out;   /* bwd: accumulated (+=), NULL = skip */
  /* activations written by fwd and read by bwd, [R][...] */
  float *theta;                     /* [R][d]   '{prefix}_theta'                  */
  float *prob;                      /* [R][L]   '{prefix}_affinity_prob'          */
  float *s;                         /* [R][dB]  sum_j p_j bp_j                    */
  float *t;                         /* [R][d]   '{prefix}_y'                      */
  float *xhat;                      /* [R][d]   LayerNorm output (t itself without PRE_ACT_LN); relu(xhat) feeds out */
  float *ln_mean, *ln_std;          /* [R]                                         */
  float *out;                       /* [R][dA]  '{prefix}_out' (before dropout)   */
  float *a_out;                     /* [R][dA]  '{prefix}_sum' = input + dropout(out) */
  uint64_t drop_offset;             /* Philox counter offset of this layer's dropout (vlfb_dropout_fwd's generator) */
} vlfb_fbo_layer_t;

typedef struct {
  int R, L;                         /* RoIs, bank rows per RoI                     */
  int dA, d, dB;                    /* query width, latent width, projected-bank width */
  int layers;                       /* 1..4                                        */
  float scale;                      /* d^-0.5 with FBO_NL.SCALE, else 1            */
  int pre_act;                      /* must be 1 (post-activation graphs keep the as-written lowering) */
  int pre_act_ln;                   /* FBO_NL.PRE_ACT_LN                           */
  float ln_eps;
  float drop_ratio;                 /* 0 = no dropout on the layer outputs         */
  uint64_t seed;
  const int64_t* step;              /* optional device scalar added to the counter (<< 32), as in vlfb_dropout_fwd */
} vlfb_fbo_cfg_t;

size_t vlfb_fbo_nl_scratch_floats(const vlfb_fbo_cfg_t* cfg);
/* a0 [R][dA] (prepare_nl_input output), bp [R][L][dB] */
int vlfb_fbo_nl_fwd(const vlfb_fbo_cfg_t* cfg, const vlfb_fbo_layer_t* layers, const float* a0, const float* bp,
                    void* stream);
/* da_last [R][dA] = gradient of the last layer's sum; writes da0 [R][dA] and dbp [R][L][dB] (overwritten) and accumulates
 * the weight / bias gradients of every layer. */
int vlfb_fbo_nl_bwd(const vlfb_fbo_cfg_t* cfg, const vlfb_fbo_layer_t* layers, const float* a0, const float* bp,
                    const float* da_last, float* da0, float* dbp, float* scratch, size_t scratch_floats, void* stream);

/* ---- device-resident feature bank: window assembly (tools/lfb_loader.py:51-152 builds the bank,
 *      lib/datasets/ava.py:300-323 / charades.py:251-276 sample a window per example) -----------
 * out[i][:] = idx[i] >= 0 ? bank[idx[i]][:] : 0 for `rows` output rows of D floats; idx is a device int32 table the
 * host fills with the reference's own sampling logic (-1 = zero padding). */
int vlfb_lfb_gather(const float* bank, int64_t bank_rows, const int32_t* idx, float* out, int64_t rows, int D,
                    int tf32_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VLFB_H_ */
