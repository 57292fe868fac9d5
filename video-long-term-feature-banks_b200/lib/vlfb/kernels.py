"""Tensor-level wrappers around the C ABI (libvlfb.so).

PyTorch tensors are used purely as device-memory containers: every function takes
CUDA fp32 tensors, validates shapes/strides and passes raw pointers to the library.
Physical layout of activations is channels-last: [N, T, H, W, C] contiguous.
"""
import ctypes as C

import torch

from . import libvlfb as L

NUM_SMS = 148


LAUNCHES = 0            # kernels launched through this module (bench.py reports it as gpu_launches)
_PROFILE = None         # when a list: (name, relaunch closure, flops, bytes, label, kept-alive operands) per profiled launch
LABEL = ''              # blob name of the graph step being executed (set by the executor; profile records carry it)


def _check(rc, what):
    global LAUNCHES
    LAUNCHES += 1
    L.check(rc, what)


def start_profile():
    """Record every tensor-core GEMM launch (its parameter block and operand tensors) until stop_profile()."""
    global _PROFILE
    _PROFILE = []


def stop_profile(reps=5):
    """Returns [(kind, milliseconds, flops, algorithmic_bytes, label)] of the GEMM launches since start_profile().
    milliseconds = DEVICE time of the launch: each recorded launch is replayed `reps` times back to back on the
    stream between two CUDA events (after one warm-up replay), so the host's launch latency -- which dominates an
    eager step of ~600 short kernels -- is not in the number.  The replays re-run the same parameter block on the
    same (kept-alive) operands; accumulating launches therefore leave garbage in their outputs: profile LAST.
    algorithmic bytes = every operand / result tensor of the launch once (the im2col expansion is not counted)."""
    global _PROFILE, LAUNCHES
    recs, _PROFILE = _PROFILE, None
    torch.cuda.synchronize()
    out = []
    n0 = LAUNCHES
    for name, relaunch, flops, nbytes, label, _keep in (recs or []):
        L.check(relaunch(), name + ' (profile replay)')
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            relaunch()
        e.record()
        e.synchronize()
        out.append((name, s.elapsed_time(e) / reps, flops, nbytes, label))
    LAUNCHES = n0
    return out


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    if t is None:
        return None
    assert t.is_cuda, 'vlfb kernels need CUDA tensors (there is no CPU fallback)'
    return C.c_void_p(t.data_ptr())


def _f32c(t, name='tensor'):
    assert t.dtype == torch.float32 and t.is_contiguous(), '%s must be contiguous fp32' % name
    return t


# Per-call execution options of vlfb_gemm (vlfb_gemm_params_t.engine / tile_n / pair / stream_k): host-side settings of
# THIS module, copied into every parameter block -- the library itself keeps no mutable state.
_ENGINE = L.ENGINE_TCGEN05
GEMM_OPTS = {'tile_n': 0, 'pair': 0, 'stream_k': 0}       # 0 = library default; tests / tuning scripts override
_GEMM_WS = {}                                             # device index -> stream-K workspace tensor


def set_gemm_backend(name):
    """'tcgen05' (default) or 'simt' (debug cross-check engine)."""
    global _ENGINE
    _ENGINE = {'tcgen05': L.ENGINE_TCGEN05, 'simt': L.ENGINE_SIMT}[name]


def get_gemm_backend():
    return ['tcgen05', 'simt'][_ENGINE]


def gemm_workspace(device):
    """Stream-K scratch of vlfb_gemm (partial tiles + arrival counters): one zero-filled buffer per device, shared
    by every launch (they are stream-ordered; the kernel leaves the counters zeroed)."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    ws = _GEMM_WS.get(idx)
    if ws is None:
        ws = torch.zeros(int(L.load().vlfb_gemm_workspace_bytes()) // 4, dtype=torch.float32, device=device)
        _GEMM_WS[idx] = ws
    return ws


# --------------------------------------------------------------------------- geometry
def conv_geom(in_shape, cout, kernels, strides, pads, dilations=(1, 1, 1)):
    """in_shape = physical (N,T,H,W,C).  Output extents follow Caffe2 Conv/Pool (floor)."""
    n, t, h, w, c = [int(v) for v in in_shape]
    g = L.ConvGeom()
    g.N, g.T, g.H, g.W, g.C = n, t, h, w, c
    g.kT, g.kH, g.kW = [int(v) for v in kernels]
    g.sT, g.sH, g.sW = [int(v) for v in strides]
    g.pT, g.pH, g.pW = [int(v) for v in pads]
    g.dT, g.dH, g.dW = [int(v) for v in dilations]
    g.To = (t + 2 * g.pT - g.dT * (g.kT - 1) - 1) // g.sT + 1
    g.Ho = (h + 2 * g.pH - g.dH * (g.kH - 1) - 1) // g.sH + 1
    g.Wo = (w + 2 * g.pW - g.dW * (g.kW - 1) - 1) // g.sW + 1
    g.Co = int(cout)
    return g


def out_shape(g):
    return (g.N, g.To, g.Ho, g.Wo, g.Co)


def _is_pointwise(g):
    return (g.kT, g.kH, g.kW, g.sT, g.sH, g.sW, g.pT, g.pH, g.pW) == (1, 1, 1, 1, 1, 1, 0, 0, 0)


def _operand(ptr_t, kind, ld=0, batch_stride=0):
    o = L.Operand()
    o.ptr = ptr_t.data_ptr()
    o.kind = kind
    o.ld = int(ld)
    o.batch_stride = int(batch_stride)
    return o


def _stem_pitch(x, g):
    """conv1 input [N,T,H,W,4]: dense, or a view of a W-padded buffer [N,T,H,pitch,4] (zero pad pixels; workspace feeds
    the clip that way so that the stem operand is staged by TMA).  Returns the row pitch in pixels."""
    assert x.dtype == torch.float32 and x.shape[-1] == 4 and x.stride(4) == 1 and x.stride(3) == 4
    pitch = x.stride(2) // 4
    assert x.stride(2) == pitch * 4 and pitch >= g.W
    assert x.stride(1) == pitch * 4 * g.H and (g.N == 1 or x.stride(0) == pitch * 4 * g.H * g.T), \
        'stem input must be [N,T,H,W,4] with padded rows only'
    return pitch


def _nbytes(*ts):
    return float(sum(t.numel() * t.element_size() for t in ts if t is not None))


def _run_gemm(p, kind='gemm', flops=None, nbytes=0.0, keep=()):
    _check(L.load().vlfb_gemm(C.byref(p), _stream()), 'vlfb_gemm')
    if _PROFILE is not None:
        if flops is None:
            flops = 2.0 * p.M * p.N * p.K * max(p.batch, 1) * max(p.taps, 1)
        q = L.GemmParams()
        C.memmove(C.byref(q), C.byref(p), C.sizeof(L.GemmParams))
        lib, st = L.load(), _stream()
        _PROFILE.append(('%s M=%d N=%d K=%d z=%d%s' % (kind, p.M, p.N, p.K, max(p.batch, p.taps),
                                                      'xauto' if p.split_k == 0 else ''),
                         lambda: lib.vlfb_gemm(C.byref(q), st), flops, nbytes, LABEL, keep))


def _base_params(M, N, K, d, ldd, alpha=1.0):
    p = L.GemmParams()
    p.M, p.N, p.K = int(M), int(N), int(K)
    p.batch, p.taps, p.split_k = 1, 1, 1
    p.d = d.data_ptr()
    p.ldd = int(ldd)
    p.d_batch_stride = 0
    p.d_tap_stride = 0
    p.alpha = float(alpha)
    p.flags = 0
    p.engine = _ENGINE
    p.tile_n, p.pair, p.stream_k = GEMM_OPTS['tile_n'], GEMM_OPTS['pair'], GEMM_OPTS['stream_k']
    ws = gemm_workspace(d.device)
    p.workspace = ws.data_ptr()
    p.workspace_bytes = ws.numel() * 4
    return p


def _set_epilogue(p, scale=None, bias=None, row_scale=None, residual=None, relu=False, tf32=False):
    keep = []
    if tf32:
        p.flags |= L.EPI_TF32
    if scale is not None:
        p.col_scale = _f32c(scale).data_ptr()
    if bias is not None:
        p.col_bias = _f32c(bias).data_ptr()
    if row_scale is not None:
        p.row_scale = _f32c(row_scale).data_ptr()
    if residual is not None:
        p.residual = _f32c(residual).data_ptr()
    if relu:
        p.flags |= L.EPI_RELU
    return keep


# --------------------------------------------------------------------------- convolution
def conv_fwd(x, w, y, g, scale=None, bias=None, residual=None, relu=False, tf32_out=False, relu_bits=None):
    """y = epi(conv(x, w)).  x [N,T,H,W,C], w [Co,kT,kH,kW,C], y [N,To,Ho,Wo,Co];
    epi: *scale[co] + bias[co] (+ residual) (ReLU).  C == 4 selects the stem (conv1) path with
    w [Co,kT,kH,8,4].  relu_bits (int32 [y.numel() / 32], with relu): also the sign bits of y, the mask of the
    ReLU's backward (conv_dgrad relu_mask_bits)."""
    _f32c(w, 'w'), _f32c(y, 'y')
    assert tuple(x.shape) == (g.N, g.T, g.H, g.W, g.C) and tuple(y.shape) == out_shape(g)
    M = g.N * g.To * g.Ho * g.Wo
    if g.C == 4:
        K = g.kT * g.kH * 32
        assert tuple(w.shape) == (g.Co, g.kT, g.kH, 8, 4)
        a = _operand(x, L.OP_STEM_K, ld=_stem_pitch(x, g))
    elif _is_pointwise(g):
        K = g.C
        a = _operand(_f32c(x, 'x'), L.OP_DENSE_K, ld=g.C)
    else:
        K = g.kT * g.kH * g.kW * g.C
        assert tuple(w.shape) == (g.Co, g.kT, g.kH, g.kW, g.C)
        a = _operand(_f32c(x, 'x'), L.OP_CONV_K)
    p = _base_params(M, g.Co, K, y, g.Co)
    p.a = a
    p.b = _operand(w, L.OP_DENSE_K, ld=K)
    p.g = g
    _set_epilogue(p, scale, bias, None, residual, relu, tf32_out)
    if relu_bits is not None:
        assert relu and relu_bits.dtype == torch.int32 and relu_bits.numel() * 32 == y.numel() and relu_bits.is_contiguous()
        p.relu_bits_out = relu_bits.data_ptr()
    _run_gemm(p, 'conv_fwd', 2.0 * M * g.Co * g.kT * g.kH * g.kW * (3 if g.C == 4 else g.C),
              _nbytes(x, w, y, residual) + (relu_bits.numel() * 4.0 if relu_bits is not None else 0.0),
              keep=(x, w, y, scale, bias, residual, relu_bits))


def conv_dgrad(dy, wt, dx, g, accumulate=False, residual=None, relu_mask=None, tf32_out=False, relu_mask_bits=None):
    """dx = finish(conv_transpose(dy, w) [+ dx if accumulate] [+ residual]).  wt [C, kT,kH,kW, Co] (see
    weight_transpose), dx [N,T,H,W,C].  finish = the backward of the ReLU that produced this layer's input
    (relu_mask = that activation, dx zeroed where it is <= 0) and the TF32 rounding the next GEMM needs: when
    this GEMM is the last contribution to the gradient, both are done here instead of in two more passes."""
    _f32c(dy, 'dy'), _f32c(wt, 'wt'), _f32c(dx, 'dx')
    assert tuple(dy.shape) == out_shape(g) and tuple(dx.shape) == (g.N, g.T, g.H, g.W, g.C)
    M = g.N * g.T * g.H * g.W
    if _is_pointwise(g):
        K = g.Co
        a = _operand(dy, L.OP_DENSE_K, ld=g.Co)
    else:
        K = g.kT * g.kH * g.kW * g.Co
        a = _operand(dy, L.OP_DGRAD_K)
    p = _base_params(M, g.C, K, dx, g.C)
    p.a = a
    p.b = _operand(wt, L.OP_DENSE_K, ld=K)
    p.g = g
    if accumulate:
        p.flags |= L.EPI_ACCUM
    if residual is not None:
        assert tuple(residual.shape) == tuple(dx.shape)
        p.residual = _f32c(residual, 'residual').data_ptr()
    if relu_mask is not None:
        assert tuple(relu_mask.shape) == tuple(dx.shape) and relu_mask_bits is None
        p.relu_mask = _f32c(relu_mask, 'relu_mask').data_ptr()
    if relu_mask_bits is not None:          # the same mask as sign bits (conv_fwd relu_bits / relu_bits): 1/32 of the bytes
        assert relu_mask_bits.dtype == torch.int32 and relu_mask_bits.numel() * 32 == dx.numel()
        p.relu_mask_bits = relu_mask_bits.data_ptr()
    if tf32_out:
        p.flags |= L.EPI_TF32
    # algorithmic dgrad work = forward MACs of the same layer
    _run_gemm(p, 'conv_dgrad', 2.0 * g.N * g.To * g.Ho * g.Wo * g.Co * g.kT * g.kH * g.kW * g.C,
              _nbytes(dy, wt, dx, residual, relu_mask) + (_nbytes(dx) if accumulate else 0.0) +
              (relu_mask_bits.numel() * 4.0 if relu_mask_bits is not None else 0.0),
              keep=(dy, wt, dx, residual, relu_mask, relu_mask_bits))


def conv_wgrad(dy, x, dw, g, row_scale=None, col_mask=None):
    """dw[co,tap,ci] += row_scale[co] * sum_m dy[m,co] * x[gather(m,tap),ci]  (atomic accumulate:
    dw must be zero-initialised or hold a partial sum).  Stem path when C == 4 (dw [Co,kT,kH,8,4],
    col_mask [32] zeroes the padding lanes)."""
    _f32c(dy, 'dy'), _f32c(dw, 'dw')
    Kpos = g.N * g.To * g.Ho * g.Wo
    if g.C == 4:
        taps, n = g.kT, g.kH * 32
        b = _operand(x, L.OP_STEM_MN, ld=_stem_pitch(x, g))
        if col_mask is not None and col_mask.numel() == 32:
            col_mask = col_mask.repeat(g.kH)
    elif _is_pointwise(g):
        taps, n = 1, g.C
        b = _operand(_f32c(x, 'x'), L.OP_DENSE_MN, ld=g.C)
    else:
        taps, n = g.kT, g.kH * g.kW * g.C          # one z-slice per temporal tap; N spans (kh, kw, ci)
        b = _operand(_f32c(x, 'x'), L.OP_CONV_MN)
    p = _base_params(g.Co, n, Kpos, dw, taps * n)
    p.a = _operand(dy, L.OP_DENSE_MN, ld=g.Co)
    p.b = b
    p.g = g
    p.taps = taps
    p.d_tap_stride = n
    p.split_k = 0            # split-K and the tile width are chosen together by the library (gemm_tc.cu launch())
    p.flags |= L.EPI_ATOMIC
    _set_epilogue(p, col_mask, None, row_scale, None, False)
    _run_gemm(p, 'conv_wgrad', 2.0 * Kpos * g.Co * g.kT * g.kH * g.kW * (3 if g.C == 4 else g.C),
              _nbytes(dy, x, dw), keep=(dy, x, dw, row_scale, col_mask))


def weight_transpose(w, wt, scale=None):
    """wt[ci][tap][co] = w[co][tap][ci] * scale[co]."""
    _f32c(w), _f32c(wt)
    co, ci = w.shape[0], w.shape[-1]
    taps = w.numel() // (co * ci)
    _check(L.load().vlfb_weight_transpose(_ptr(w), _ptr(wt), _ptr(scale), co, taps, ci, _stream()),
            'weight_transpose')


# --------------------------------------------------------------------------- generic matmul
def _dim_ok(stride, size):
    return size == 1 or stride == 1


def _mat_operand(t, rows_dim, k_dim):
    """Describe logical matrix op[row,k] = t[..., row(s), k(s)] (3-D strided view, dim 0 = batch)."""
    sb, sr, sk = t.stride(0), t.stride(rows_dim), t.stride(k_dim)
    R, K = t.shape[rows_dim], t.shape[k_dim]
    if t.shape[0] == 1:
        sb = 0
    k_ok, mn_ok = _dim_ok(sk, K), _dim_ok(sr, R)
    k_al = (R == 1 or sr % 4 == 0) and K % 4 == 0 and sb % 4 == 0       # 16-byte addressable for tcgen05
    mn_al = (K == 1 or sk % 4 == 0) and R % 4 == 0 and sb % 4 == 0
    if k_ok and (k_al or not (mn_ok and mn_al)):
        return L.OP_DENSE_K, (sr if R > 1 else K), sb
    if mn_ok:
        return L.OP_DENSE_MN, (sk if K > 1 else R), sb       # unaligned cases run on the SIMT engine (api.cu)
    raise ValueError('matmul operand with shape %s strides %s is not tensor-core addressable'
                     % (tuple(t.shape), tuple(t.stride())))


def matmul(a, b, d, alpha=1.0, accumulate=False, bias=None, tf32_out=False, tf32_optional=False):
    """d[i] (+)= alpha * a[i] @ b[i] (+ bias[n]) for 3-D strided views a (B,M,K), b (B,K,N), d (B,M,N).
    Each matrix needs unit stride along one of its two dims (16-byte aligned rows).  Returns whether d was stored
    TF32-rounded: with `tf32_optional` a product that qualifies for split-K (atomic accumulation cannot round) keeps
    the split and leaves the rounding to the consumer -- the split is worth 2x on the K = 3136 non-local gradient
    products, the saved rounding pass ~5 us (call J/K: 0.046 vs 0.022 ms per launch)."""
    assert a.dim() == 3 and b.dim() == 3 and d.dim() == 3
    Bt, M, K = a.shape
    N = b.shape[2]
    assert b.shape[0] == Bt and b.shape[1] == K and tuple(d.shape) == (Bt, M, N)
    if not _dim_ok(d.stride(2), N):
        # output is column-major: compute d^T = b^T a^T
        assert _dim_ok(d.stride(1), M), 'matmul output needs a unit stride'
        assert bias is None
        return matmul(b.transpose(1, 2), a.transpose(1, 2), d.transpose(1, 2), alpha, accumulate, None, tf32_out,
                      tf32_optional)
    ka, lda, sba = _mat_operand(a, 1, 2)
    kb, ldb, sbb = _mat_operand(b, 2, 1)
    p = _base_params(M, N, K, d, d.stride(1) if M > 1 else N, alpha)
    p.a = _operand(a, ka, lda, sba)
    p.b = _operand(b, kb, ldb, sbb)
    p.batch = Bt
    p.d_batch_stride = d.stride(0) if Bt > 1 else 0
    tiles = Bt * ((M + 127) // 128) * ((N + 255) // 256)
    if tiles <= NUM_SMS // 2 and K >= 1024 and tf32_out and tf32_optional:
        tf32_out = False
    if tiles <= NUM_SMS // 2 and K >= 1024 and not tf32_out:
        # few output tiles with a long reduction (the 4 x 80 x 2560 classifier ran 0.19 ms on ONE CTA; the non-local
        # affinity products fill 28-56 of 148 SMs): split K over the SMs -- atomic accumulation into a zeroed / kept
        # D, bias from the first slice; the library picks the split together with the tile width
        if not accumulate:
            fill(d, 0.0) if d.is_contiguous() else d.zero_()
        p.split_k = 0
        p.flags |= L.EPI_ATOMIC
    elif accumulate:
        p.flags |= L.EPI_ACCUM
    _set_epilogue(p, None, bias, None, None, False, tf32_out)
    _run_gemm(p, 'matmul', 2.0 * Bt * M * N * K, 4.0 * Bt * (M * K + K * N + M * N * (2 if accumulate else 1)),
              keep=(a, b, d, bias))
    return bool(tf32_out)


def weight_transpose_multi(jobs, cache):
    """jobs = [(w, wt, scale_or_None)]: every dgrad weight operand of the step in one launch.  The device job
    table is built once and kept in `cache` (all addresses are static: parameters and persistent wt buffers)."""
    import numpy as np
    key = tuple((w.data_ptr(), wt.data_ptr(), 0 if s is None else s.data_ptr()) for w, wt, s in jobs)
    if cache.get('key') != key:
        dt = np.dtype([('w', '<u8'), ('wt', '<u8'), ('scale', '<u8'), ('co', '<i4'), ('taps', '<i4'), ('ci', '<i4'),
                       ('bb', '<i4')])
        tab = np.zeros(len(jobs), dtype=dt)
        blocks = 0
        for i, (w, wt, s) in enumerate(jobs):
            _f32c(w), _f32c(wt)
            co, ci = w.shape[0], w.shape[-1]
            taps = w.numel() // (co * ci)
            tab[i] = (w.data_ptr(), wt.data_ptr(), 0 if s is None else s.data_ptr(), co, taps, ci, blocks)
            blocks += ((ci + 31) // 32) * ((co + 31) // 32) * taps
        assert tab.dtype.itemsize == 40
        cache['table'] = torch.from_numpy(tab.view(np.uint8).copy()).to(jobs[0][0].device)
        cache['blocks'] = blocks
        cache['key'] = key
    _check(L.load().vlfb_weight_transpose_multi(_ptr(cache['table']), len(jobs), cache['blocks'], _stream()),
           'weight_transpose_multi')


# --------------------------------------------------------------------------- streaming ops
def affine_fwd(x, s, b, y):
    _check(L.load().vlfb_affine_nd_fwd(_ptr(_f32c(x)), _ptr(s), _ptr(b), _ptr(_f32c(y)),
                                        x.numel() // x.shape[-1], x.shape[-1], _stream()), 'affine_fwd')


def affine_bwd(dy, s, dx):
    _check(L.load().vlfb_affine_nd_bwd(_ptr(_f32c(dy)), _ptr(s), _ptr(_f32c(dx)),
                                        dy.numel() // dy.shape[-1], dy.shape[-1], _stream()), 'affine_bwd')


def _bn_workspace(C_):
    nbytes = int(L.load().vlfb_spatial_bn_workspace_bytes(int(C_)))
    return torch.empty((nbytes + 15) // 16 * 16, dtype=torch.uint8, device='cuda'), nbytes


def spatial_bn_fwd(x, s, b, rm, rv, sm, siv, y, eps, momentum):
    """Training-mode SpatialBN of a channels-last [..., C] tensor: batch statistics -> sm / siv (saved mean, inverse std),
    running statistics rm / rv updated in place (None: left alone), y = normalised * s + b."""
    ws, nb = _bn_workspace(x.shape[-1])
    _check(L.load().vlfb_spatial_bn_fwd(_ptr(_f32c(x)), _ptr(s), _ptr(b), _ptr(rm), _ptr(rv), _ptr(sm), _ptr(siv),
                                        _ptr(_f32c(y)), x.numel() // x.shape[-1], x.shape[-1], float(eps), float(momentum),
                                        _ptr(ws), nb, _stream()), 'spatial_bn_fwd')


def spatial_bn_infer(x, s, b, rm, rv, y, eps):
    ws, nb = _bn_workspace(x.shape[-1])
    _check(L.load().vlfb_spatial_bn_infer(_ptr(_f32c(x)), _ptr(s), _ptr(b), _ptr(rm), _ptr(rv), _ptr(_f32c(y)),
                                          x.numel() // x.shape[-1], x.shape[-1], float(eps), _ptr(ws), nb, _stream()),
           'spatial_bn_infer')


def spatial_bn_bwd(dy, x, s, sm, siv, dx, ds, db):
    """dx of training-mode SpatialBN; ds += sum dy * xhat, db += sum dy (either may be None)."""
    ws, nb = _bn_workspace(x.shape[-1])
    _check(L.load().vlfb_spatial_bn_bwd(_ptr(_f32c(dy)), _ptr(_f32c(x)), _ptr(s), _ptr(sm), _ptr(siv), _ptr(_f32c(dx)),
                                        _ptr(ds), _ptr(db), x.numel() // x.shape[-1], x.shape[-1], _ptr(ws), nb, _stream()),
           'spatial_bn_bwd')


def maxpool_fwd(x, y, argmax, g):
    _check(L.load().vlfb_maxpool3d_fwd(_ptr(_f32c(x)), _ptr(_f32c(y)), _ptr(argmax), C.byref(g), _stream()),
            'maxpool_fwd')


def maxpool_bwd(dy, argmax, dx, g):
    _check(L.load().vlfb_maxpool3d_bwd(_ptr(_f32c(dy)), _ptr(argmax), _ptr(_f32c(dx)), C.byref(g), _stream()),
            'maxpool_bwd')


def maxpool_bwd_gather(dy, argmax, y, dx, g, tf32_out=False):
    """dx = max-pool backward in gather form (every element written once: no fill, no atomics); y = the pool output
    (or None): windows with a maximum <= 0 pass nothing (the backward of the ReLU feeding the pool)."""
    _check(L.load().vlfb_maxpool3d_bwd_gather(_ptr(_f32c(dy)), _ptr(argmax), _ptr(y), _ptr(_f32c(dx)), C.byref(g),
                                              int(tf32_out), _stream()), 'maxpool_bwd_gather')


def avgpool_fwd(x, y, g):
    _check(L.load().vlfb_avgpool3d_fwd(_ptr(_f32c(x)), _ptr(_f32c(y)), C.byref(g), _stream()), 'avgpool_fwd')


def avgpool_bwd(dy, dx, g, accumulate=False):
    _check(L.load().vlfb_avgpool3d_bwd(_ptr(_f32c(dy)), _ptr(_f32c(dx)), C.byref(g), int(accumulate), _stream()),
            'avgpool_bwd')


def roi_align_fwd(feat, rois, out, spatial_scale, sampling_ratio=0):
    """feat [N,H,W,C], rois [R,5], out [R,PH,PW,C]."""
    n, h, w, c = feat.shape
    r, ph, pw, _ = out.shape
    _check(L.load().vlfb_roi_align_fwd(_ptr(_f32c(feat)), _ptr(_f32c(rois)), _ptr(_f32c(out)), n, h, w, c, r, ph, pw,
                                        float(spatial_scale), int(sampling_ratio), _stream()), 'roi_align_fwd')


def roi_align_bwd(dout, rois, dfeat, spatial_scale, sampling_ratio=0):
    n, h, w, c = dfeat.shape
    r, ph, pw, _ = dout.shape
    _check(L.load().vlfb_roi_align_bwd(_ptr(_f32c(dout)), _ptr(_f32c(rois)), _ptr(_f32c(dfeat)), n, h, w, c, r, ph,
                                        pw, float(spatial_scale), int(sampling_ratio), _stream()), 'roi_align_bwd')


def roi_align_table(rois, h, w, ph, pw, max_grid, spatial_scale, sampling_ratio=0):
    r = rois.shape[0]
    pos = torch.empty((r, ph, pw, max_grid, max_grid, 4), dtype=torch.int32, device=rois.device)
    wts = torch.empty((r, ph, pw, max_grid, max_grid, 4), dtype=torch.float32, device=rois.device)
    grid = torch.empty((r, 2), dtype=torch.int32, device=rois.device)
    _check(L.load().vlfb_roi_align_table(_ptr(_f32c(rois)), _ptr(pos), _ptr(wts), _ptr(grid), h, w, r, ph, pw,
                                          max_grid, float(spatial_scale), int(sampling_ratio), _stream()),
            'roi_align_table')
    return pos, wts, grid


def softmax_fwd(x, p, scale=1.0, tf32_out=False):
    cols = x.shape[-1]
    _check(L.load().vlfb_softmax_fwd(_ptr(_f32c(x)), _ptr(_f32c(p)), x.numel() // cols, cols, float(scale),
                                      int(tf32_out), _stream()), 'softmax_fwd')


def softmax_bwd(p, dp, dx, scale=1.0, tf32_out=False):
    cols = p.shape[-1]
    _check(L.load().vlfb_softmax_bwd(_ptr(_f32c(p)), _ptr(_f32c(dp)), _ptr(_f32c(dx)), p.numel() // cols, cols,
                                      float(scale), 1 if tf32_out else 0, _stream()), 'softmax_bwd')


def layernorm_fwd(x, y, mean, std, cols, eps=1e-5):
    _check(L.load().vlfb_layernorm_fwd(_ptr(_f32c(x)), _ptr(_f32c(y)), _ptr(mean), _ptr(std), x.numel() // cols,
                                        cols, float(eps), _stream()), 'layernorm_fwd')


def layernorm_bwd(dy, y, std, dx, cols):
    _check(L.load().vlfb_layernorm_bwd(_ptr(_f32c(dy)), _ptr(_f32c(y)), _ptr(std), _ptr(_f32c(dx)),
                                        dy.numel() // cols, cols, _stream()), 'layernorm_bwd')


def relu_fwd(x, y):
    _check(L.load().vlfb_relu_fwd(_ptr(_f32c(x)), _ptr(_f32c(y)), x.numel(), _stream()), 'relu_fwd')


def relu_bwd(dy, y, dx):
    _check(L.load().vlfb_relu_bwd(_ptr(_f32c(dy)), _ptr(_f32c(y)), _ptr(_f32c(dx)), dy.numel(), _stream()),
            'relu_bwd')


def axpby(x, a, y, b, out):
    """out = a*x + b*y (y may be None when b == 0)."""
    _check(L.load().vlfb_axpby(_ptr(_f32c(x)), float(a), _ptr(y), float(b), _ptr(_f32c(out)), x.numel(),
                                _stream()), 'axpby')


def fill(x, v):
    _check(L.load().vlfb_fill(_ptr(_f32c(x)), float(v), x.numel(), _stream()), 'fill')


def round_tf32(x, y):
    _check(L.load().vlfb_round_tf32(_ptr(_f32c(x)), _ptr(_f32c(y)), x.numel(), _stream()), 'round_tf32')


def add_tf32(x, y, out):
    _check(L.load().vlfb_add_tf32(_ptr(_f32c(x)), _ptr(_f32c(y)), _ptr(_f32c(out)), x.numel(), _stream()), 'add_tf32')


def relu_tf32(x, y):
    _check(L.load().vlfb_relu_tf32(_ptr(_f32c(x)), _ptr(_f32c(y)), x.numel(), _stream()), 'relu_tf32')


def add_relu_bwd_tf32(a, b, y, out):
    """out = (y is None or y > 0) ? round_tf32(a + b) : 0 (one pass; out may alias a or b)."""
    _check(L.load().vlfb_add_relu_bwd_tf32(_ptr(_f32c(a)), _ptr(_f32c(b)), _ptr(y), _ptr(_f32c(out)), a.numel(),
                                            _stream()), 'add_relu_bwd_tf32')


def relu_bits(x, bits):
    """bits (int32 [x.numel() / 32]): bit e = x.flat[e] > 0."""
    assert bits.dtype == torch.int32 and bits.numel() * 32 == x.numel()
    _check(L.load().vlfb_relu_bits(_ptr(_f32c(x)), bits.data_ptr(), x.numel(), _stream()), 'relu_bits')


def relu_bwd_tf32(dy, y, dx):
    _check(L.load().vlfb_relu_bwd_tf32(_ptr(_f32c(dy)), _ptr(_f32c(y)), _ptr(_f32c(dx)), dy.numel(), _stream()),
           'relu_bwd_tf32')


def colsum(x, ld, out, rows, cols, accumulate=False):
    lib = L.load()
    nbytes = int(lib.vlfb_colsum_workspace_bytes(int(rows), int(cols)))
    ws = torch.empty(max(nbytes // 4, 1), dtype=torch.float32, device=out.device)     # slab partial sums
    _check(lib.vlfb_colsum(_ptr(x), int(ld), _ptr(out), int(rows), int(cols), int(accumulate), _ptr(ws), nbytes,
                           _stream()), 'colsum')


def sigmoid_fwd(x, y):
    _check(L.load().vlfb_sigmoid_fwd(_ptr(_f32c(x)), _ptr(_f32c(y)), x.numel(), _stream()), 'sigmoid_fwd')


def dropout(x, y, ratio, seed, offset, step=None):
    """y = x * mask / (1-ratio); the mask is a pure function of (seed, offset, index), so the same
    call on dy is the backward."""
    _check(L.load().vlfb_dropout_fwd(_ptr(_f32c(x)), _ptr(_f32c(y)), x.numel(), float(ratio), int(seed),
                                      int(offset), _ptr(step), _stream()), 'dropout')


def copy2d(src, lds, dst, ldd, rows, cols, accumulate=False, src_off=0, dst_off=0):
    sp = C.c_void_p(src.data_ptr() + 4 * src_off)
    dp = C.c_void_p(dst.data_ptr() + 4 * dst_off)
    _check(L.load().vlfb_copy2d(sp, int(lds), dp, int(ldd), int(rows), int(cols), int(accumulate), _stream()),
            'copy2d')


def nc_to_cl(src, dst, n, c, inner, cpad=None, tf32_out=False, width=0, pitch=0, left=0):
    """NCTHW -> NDHWC (C padded to cpad).  width / pitch / left: the destination rows are `pitch` pixels long and the
    `width` real pixels of a row start at pixel `left` (the W-padded clip of conv1's TMA path)."""
    if pitch:
        _check(L.load().vlfb_nc_to_cl_pitched(_ptr(_f32c(src)), _ptr(_f32c(dst)), n, c, inner, cpad or c, int(tf32_out),
                                              int(width), int(pitch), int(left), _stream()), 'nc_to_cl_pitched')
        return
    _check(L.load().vlfb_nc_to_cl_round(_ptr(_f32c(src)), _ptr(_f32c(dst)), n, c, inner, cpad or c, int(tf32_out),
                                        _stream()), 'nc_to_cl')


def cl_to_nc(src, dst, n, c, inner, cpad=None):
    _check(L.load().vlfb_cl_to_nc(_ptr(_f32c(src)), _ptr(_f32c(dst)), n, c, inner, cpad or c, _stream()), 'cl_to_nc')


def sigmoid_ce_fwd(logits, targets, loss, scale):
    assert targets.dtype == torch.int32
    _check(L.load().vlfb_sigmoid_ce_fwd(_ptr(_f32c(logits)), _ptr(targets), _ptr(loss), logits.numel(),
                                         float(scale), _stream()), 'sigmoid_ce_fwd')


def sigmoid_ce_bwd(logits, targets, dloss, dlogits, scale):
    _check(L.load().vlfb_sigmoid_ce_bwd(_ptr(_f32c(logits)), _ptr(targets), _ptr(dloss), _ptr(_f32c(dlogits)),
                                         logits.numel(), float(scale), _stream()), 'sigmoid_ce_bwd')


def softmax_ce_fwd(logits, labels, prob, loss, scale):
    assert labels.dtype == torch.int32
    _check(L.load().vlfb_softmax_ce_fwd(_ptr(_f32c(logits)), _ptr(labels), _ptr(_f32c(prob)), _ptr(loss),
                                         logits.shape[0], logits.shape[1], float(scale), _stream()), 'softmax_ce_fwd')


def softmax_ce_bwd(prob, labels, dlogits, scale):
    _check(L.load().vlfb_softmax_ce_bwd(_ptr(_f32c(prob)), _ptr(labels), _ptr(_f32c(dlogits)), prob.shape[0],
                                         prob.shape[1], float(scale), _stream()), 'softmax_ce_bwd')


def sgd_nesterov(p, g, m, lr, momentum, wd, nesterov=True, p_tf32=None):
    """In place: g += wd*p; m' = mu*m + lr*g; p -= (1+mu)*m' - mu*m  (lr is a 1-element device tensor)."""
    _check(L.load().vlfb_sgd_nesterov(_ptr(_f32c(p)), _ptr(_f32c(g)), _ptr(_f32c(m)), _ptr(p_tf32), p.numel(), _ptr(lr),
                                       float(momentum), float(wd), int(bool(nesterov)), _stream()), 'sgd_nesterov')


# --------------------------------------------------------------------------- training-mode FBO-NL stack (csrc/fbo.cu 3)
FBO_LAYER_KEYS = ('w_theta', 'b_theta', 'w_phi', 'b_phi', 'w_g', 'b_g', 'w_out', 'b_out',
                  'gw_theta', 'gb_theta', 'gw_phi', 'gb_phi', 'gw_g', 'gb_g', 'gw_out', 'gb_out',
                  'theta', 'prob', 's', 't', 'xhat', 'ln_mean', 'ln_std', 'out', 'a_out')


def _fbo_structs(cfgd, layers):
    c = L.FboCfg()
    for k in ('R', 'L', 'dA', 'd', 'dB'):
        setattr(c, k, int(cfgd[k]))
    c.layers = len(layers)
    c.scale, c.pre_act, c.pre_act_ln = float(cfgd['scale']), 1, int(bool(cfgd['pre_act_ln']))
    c.ln_eps, c.drop_ratio, c.seed = float(cfgd.get('ln_eps', 1e-5)), float(cfgd.get('drop_ratio', 0.0)), int(cfgd.get('seed', 0))
    step = cfgd.get('step')
    c.step = step.data_ptr() if step is not None else None
    arr = (L.FboLayer * len(layers))()
    for i, ld in enumerate(layers):
        for k in FBO_LAYER_KEYS:
            t = ld.get(k)
            if t is not None:
                _f32c(t, k)
                assert t.is_cuda
            setattr(arr[i], k, None if t is None else t.data_ptr())
        arr[i].drop_offset = int(ld.get('drop_offset', 0))
    return c, arr


def fbo_nl_fwd(cfgd, layers, a0, bp):
    """All FBO-NL layers forward in one launch.  cfgd: R, L, dA, d, dB, scale, pre_act_ln, [ln_eps, drop_ratio, seed,
    step]; layers: dicts of tensors keyed by FBO_LAYER_KEYS (weights [out][in], saved activations [R][...])."""
    _f32c(a0, 'a0'), _f32c(bp, 'bp')
    assert tuple(a0.shape) == (cfgd['R'], cfgd['dA']) and tuple(bp.shape) == (cfgd['R'], cfgd['L'], cfgd['dB'])
    c, arr = _fbo_structs(cfgd, layers)
    _check(L.load().vlfb_fbo_nl_fwd(C.byref(c), arr, _ptr(a0), _ptr(bp), _stream()), 'fbo_nl_fwd')


def fbo_nl_bwd(cfgd, layers, a0, bp, da_last, da0, dbp):
    """Backward of fbo_nl_fwd: da0, dbp (overwritten) and the accumulated weight gradients (layers[i]['gw_*'])."""
    global LAUNCHES
    for t in (a0, bp, da_last, da0, dbp):
        _f32c(t)
    c, arr = _fbo_structs(cfgd, layers)
    lib = L.load()
    n = int(lib.vlfb_fbo_nl_scratch_floats(C.byref(c)))
    scratch = torch.empty(n, dtype=torch.float32, device=a0.device)
    _check(lib.vlfb_fbo_nl_bwd(C.byref(c), arr, _ptr(a0), _ptr(bp), _ptr(da_last), _ptr(da0), _ptr(dbp), _ptr(scratch),
                               C.c_size_t(n), _stream()), 'fbo_nl_bwd')
    LAUNCHES += 1                 # two kernels (per-RoI backward + rank-R weight gradients)


# --------------------------------------------------------------------------- raw feature-bank kernels (csrc/fbo.cu)
def fbo_bank_scan(bank, q, out, scale, prob=None, tf32_out=False):
    """out[r] = sum_j softmax_j(scale * q[r].bank[r,j]) * bank[r,j]: the folded inference-mode FBO-NL layer, one pass
    over the raw bank.  bank [R,L,D] fp32 or bf16 (storage type only: the arithmetic is fp32), q [R,D], out [R,D],
    prob [R,L] or None."""
    assert bank.is_contiguous() and bank.dtype in (torch.float32, torch.bfloat16), 'bank must be contiguous fp32 / bf16'
    _f32c(q, 'q'), _f32c(out, 'out')
    dt = L.DT_BF16 if bank.dtype == torch.bfloat16 else L.DT_F32
    r, l, d = bank.shape
    assert tuple(q.shape) == (r, d) and tuple(out.shape) == (r, d)
    if prob is not None:
        assert tuple(_f32c(prob, 'prob').shape) == (r, l)
    lib = L.load()
    nbytes = int(lib.vlfb_fbo_bank_scan_workspace_dt(r, l, d, dt))
    if nbytes == 0 and r > 0:
        raise L.VlfbError('fbo_bank_scan: unsupported bank row width %d (fp32: 1024, 2048 or 4096; bf16: 2048 or 4096)' % d)
    wsp = torch.empty(max(nbytes, 4) // 4, dtype=torch.float32, device=bank.device)
    args = (_ptr(bank), dt, _ptr(q), float(scale), _ptr(out), _ptr(prob), r, l, d, int(tf32_out), _ptr(wsp),
            C.c_size_t(nbytes), _stream())
    _check(lib.vlfb_fbo_bank_scan_dt(*args), 'fbo_bank_scan')
    if _PROFILE is not None:
        _PROFILE.append(('fbo_bank_scan R=%d L=%d D=%d %s' % (r, l, d, 'bf16' if dt else 'f32'),
                         lambda: lib.vlfb_fbo_bank_scan_dt(*args), 4.0 * r * l * d, _nbytes(bank, q, out), LABEL,
                         (bank, q, out, prob, wsp)))


def cast_bf16(x, y):
    """y (bf16) = x (fp32), round to nearest even; numel % 8 == 0."""
    assert y.dtype == torch.bfloat16 and y.is_contiguous() and y.numel() == x.numel()
    _check(L.load().vlfb_cast_f32_to_bf16(_ptr(_f32c(x)), _ptr(y), x.numel(), _stream()), 'cast_bf16')


def lfb_gather(bank, idx, out, tf32_out=False):
    """out[i] = bank[idx[i]] (zeros where idx[i] < 0).  bank [rows, D] fp32, idx int32 [n], out [n, D]."""
    _f32c(bank, 'bank'), _f32c(out, 'out')
    assert idx.dtype == torch.int32 and idx.is_contiguous() and idx.is_cuda
    n, d = out.shape[0], out.shape[-1]
    assert idx.numel() == out.numel() // d and bank.shape[-1] == d
    if idx.numel() == 0:
        return
    _check(L.load().vlfb_lfb_gather(_ptr(bank), bank.numel() // d, _ptr(idx), _ptr(out), idx.numel(), d, int(tf32_out),
                                    _stream()), 'lfb_gather')
