"""GPU parity tests of the individual kernels, called through the C ABI (ctypes) and
checked against fp64 PyTorch-CPU references / the oracle.  TF32 tolerance: operands are
pre-rounded to TF32 so the tensor-core result must match fp64 to accumulation error."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from util import rel_err, stem_pack, tf32_round, to_cl, to_nc, w_to_cl

pytestmark = pytest.mark.gpu

BACKENDS = ['tcgen05', 'simt']


@pytest.fixture(scope='module')
def K():
    from vlfb import kernels
    assert torch.cuda.is_available()
    yield kernels
    kernels.set_gemm_backend('tcgen05')


def rnd(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return tf32_round(torch.randn(shape, generator=g) * scale)


# -------------------------------------------------------------------------- dense matmul
@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('M,N,K_', [(4, 80, 2560), (8, 160, 4100), (130, 36, 1024)])
def test_skinny_long_k_matmul_uses_split_k_with_bias(K, backend, M, N, K_):
    """The classifier FC (4 RoIs x 80 classes x 2560): few output tiles, long reduction -> split-K with atomic
    accumulation; the bias must be added exactly once, and accumulate=True must keep the previous contents."""
    K.set_gemm_backend(backend)
    a, b = rnd((1, M, K_), 11), rnd((1, K_, N), 12)
    bias = torch.randn(N)
    ref = torch.bmm(a.double(), b.double()) + bias.double()
    d = torch.full((1, M, N), float('nan'), device='cuda')
    K.matmul(a.cuda(), b.cuda(), d, bias=bias.cuda())
    torch.cuda.synchronize()
    assert rel_err(d, ref) < 2e-5
    K.matmul(a.cuda(), b.cuda(), d, accumulate=True)
    torch.cuda.synchronize()
    assert rel_err(d, 2 * ref - bias.double()) < 2e-5


@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('ta,tb', [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize('B,M,N,K_', [(1, 128, 128, 64), (2, 200, 80, 300), (3, 1, 300, 512), (1, 264, 512, 96),
                                       (2, 392, 196, 128)])
def test_matmul_layouts(K, backend, ta, tb, B, M, N, K_):
    K.set_gemm_backend(backend)
    if ta and M % 4:
        pytest.skip('MN-major A needs M % 4 == 0')
    if tb == 0 and N % 4:
        pytest.skip('MN-major B needs N % 4 == 0')
    a = rnd((B, K_, M) if ta else (B, M, K_), 1)
    b = rnd((B, N, K_) if tb else (B, K_, N), 2)
    A = a.transpose(1, 2) if ta else a
    Bm = b.transpose(1, 2) if tb else b
    ref = torch.bmm(A.double(), Bm.double()) * 0.5
    ad, bd = a.cuda(), b.cuda()
    d = torch.full((B, M, N), float('nan'), device='cuda')
    K.matmul(ad.transpose(1, 2) if ta else ad, bd.transpose(1, 2) if tb else bd, d, alpha=0.5)
    torch.cuda.synchronize()
    assert rel_err(d, ref) < 2e-5
    # transposed (column-major) output + accumulate
    dt = torch.ones((B, N, M), device='cuda')
    K.matmul(ad.transpose(1, 2) if ta else ad, bd.transpose(1, 2) if tb else bd, dt.transpose(1, 2), alpha=0.5,
             accumulate=True) if M % 4 == 0 and N % 4 == 0 else None
    if M % 4 == 0 and N % 4 == 0:
        torch.cuda.synchronize()
        assert rel_err(dt.transpose(1, 2), ref + 1.0) < 2e-5


def pack_sign_bits(x):
    """Reference bit layout of vlfb_gemm_params_t.relu_mask_bits / relu_bits_out: bit e & 31 of word e >> 5 = x.flat[e] > 0."""
    b = (x.reshape(-1, 32) > 0).to(torch.int64)
    v = (b << torch.arange(32, dtype=torch.int64, device=x.device)).sum(1)
    return torch.where(v >= 2 ** 31, v - 2 ** 32, v).to(torch.int32)


def test_relu_bits_kernel(K):
    x = torch.randn(7 * 4096 + 64, device='cuda')
    x[::5] = 0.0
    bits = torch.full((x.numel() // 32,), -1, dtype=torch.int32, device='cuda')
    K.relu_bits(x, bits)
    torch.cuda.synchronize()
    assert torch.equal(bits, pack_sign_bits(x))


# -------------------------------------------------------------------------- convolution
GEOMS = [
    # N, T, H, W, Ci, Co, kernels, strides, pads, dilations
    (2, 4, 8, 8, 32, 64, (3, 1, 1), (1, 1, 1), (1, 0, 0), (1, 1, 1)),
    (1, 3, 9, 10, 64, 32, (1, 3, 3), (1, 1, 1), (0, 1, 1), (1, 1, 1)),
    (2, 2, 14, 14, 32, 96, (1, 3, 3), (1, 2, 2), (0, 1, 1), (1, 1, 1)),
    (1, 2, 14, 14, 64, 64, (1, 3, 3), (1, 1, 1), (0, 2, 2), (1, 2, 2)),
    (2, 3, 6, 6, 64, 160, (1, 1, 1), (1, 1, 1), (0, 0, 0), (1, 1, 1)),
    (2, 2, 8, 8, 32, 64, (1, 1, 1), (1, 2, 2), (0, 0, 0), (1, 1, 1)),
    (1, 4, 7, 7, 256, 288, (3, 1, 1), (1, 1, 1), (1, 0, 0), (1, 1, 1)),
    # strided dgrads: parity-class decomposition on the tensor-core engine (several M tiles with a ragged tail, a temporal
    # kernel, one strided dimension only) and the gather fallback (odd extents)
    (2, 2, 30, 30, 64, 128, (1, 3, 3), (1, 2, 2), (0, 1, 1), (1, 1, 1)),
    (1, 4, 12, 16, 64, 64, (3, 3, 3), (1, 2, 2), (1, 1, 1), (1, 1, 1)),
    (1, 2, 8, 8, 32, 32, (1, 3, 3), (1, 2, 1), (0, 1, 1), (1, 1, 1)),
    (3, 2, 20, 12, 128, 64, (1, 1, 1), (1, 2, 2), (0, 0, 0), (1, 1, 1)),
    (1, 2, 15, 15, 32, 64, (1, 3, 3), (1, 2, 2), (0, 1, 1), (1, 1, 1)),
]


def _conv_ref(x, w, strides, pads, dil):
    return F.conv3d(x.double(), w.double(), None, strides, pads, dil)


@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('geom', GEOMS)
def test_conv_fwd_dgrad_wgrad(K, backend, geom):
    K.set_gemm_backend(backend)
    N, T, H, W, Ci, Co, ker, st, pd, dil = geom
    x = rnd((N, Ci, T, H, W), 3)
    w = rnd((Co, Ci) + ker, 4, 0.1)
    s = torch.rand(Co) + 0.5
    b = torch.randn(Co) * 0.1
    xd = x.double().requires_grad_(True)
    wd = w.double().requires_grad_(True)
    y = F.conv3d(xd, wd, None, st, pd, dil)
    res = rnd(tuple(y.shape), 5)
    out_ref = torch.relu(y * s.double().view(1, -1, 1, 1, 1) + b.double().view(1, -1, 1, 1, 1) + res.double())
    g = K.conv_geom((N, T, H, W, Ci), Co, ker, st, pd, dil)
    assert K.out_shape(g) == (N, y.shape[2], y.shape[3], y.shape[4], Co)
    x_cl, w_cl = to_cl(x).cuda(), w_to_cl(w).cuda()
    yd = torch.full(K.out_shape(g), float('nan'), device='cuda')
    K.conv_fwd(x_cl, w_cl, yd, g, scale=s.cuda(), bias=b.cuda(), residual=to_cl(res).cuda(), relu=True)
    torch.cuda.synchronize()
    assert rel_err(to_nc(yd), out_ref) < 2e-5
    # ... and with the sign bits of the result (the ReLU-backward mask): same values, bits exact
    yb = torch.full(K.out_shape(g), float('nan'), device='cuda')
    ybits = torch.full((yb.numel() // 32,), 0x5A5A5A5A, dtype=torch.int32, device='cuda')
    K.conv_fwd(x_cl, w_cl, yb, g, scale=s.cuda(), bias=b.cuda(), residual=to_cl(res).cuda(), relu=True, relu_bits=ybits)
    torch.cuda.synchronize()
    assert torch.equal(yb, yd) and torch.equal(ybits, pack_sign_bits(yd))
    # plain (no epilogue) forward
    K.conv_fwd(x_cl, w_cl, yd, g)
    torch.cuda.synchronize()
    assert rel_err(to_nc(yd), y) < 2e-5
    # backward
    dy = rnd(tuple(y.shape), 6)
    y.backward(dy.double())
    dy_cl = to_cl(dy).cuda()
    taps = ker[0] * ker[1] * ker[2]
    wt = torch.empty((Ci, taps, Co), device='cuda')
    K.weight_transpose(w_cl, wt)
    torch.cuda.synchronize()
    assert torch.equal(wt.cpu(), w_to_cl(w).reshape(Co, taps, Ci).permute(2, 1, 0))
    dx = torch.full((N, T, H, W, Ci), float('nan'), device='cuda')
    K.conv_dgrad(dy_cl, wt, dx, g)
    torch.cuda.synchronize()
    assert rel_err(to_nc(dx), xd.grad) < 2e-5
    K.conv_dgrad(dy_cl, wt, dx, g, accumulate=True)
    torch.cuda.synchronize()
    assert rel_err(to_nc(dx), 2 * xd.grad) < 2e-5
    # fused "gradient finish": (+ residual | + previous dx), ReLU mask by the layer input, TF32 rounding
    res = rnd((N, T, H, W, Ci), 8).cuda()
    mask = rnd((N, T, H, W, Ci), 9).cuda()
    want = to_nc((to_cl(xd.grad.float()).cuda() + res) * (mask > 0))
    dx2 = torch.full((N, T, H, W, Ci), float('nan'), device='cuda')
    K.conv_dgrad(dy_cl, wt, dx2, g, residual=res, relu_mask=mask, tf32_out=True)
    torch.cuda.synchronize()
    assert rel_err(to_nc(dx2), want) < 6e-4                          # one TF32 rounding of the result
    assert (dx2.view(torch.int32) & 0x1FFF).eq(0).all()              # low 13 mantissa bits cleared
    assert (dx2[mask <= 0] == 0).all()
    dx3 = res.clone()
    K.conv_dgrad(dy_cl, wt, dx3, g, accumulate=True, relu_mask=mask, tf32_out=True)
    torch.cuda.synchronize()
    assert torch.equal(dx3, dx2)
    # the same mask as sign bits: identical results (plain, accumulate)
    mbits = pack_sign_bits(mask)
    dx4 = torch.full((N, T, H, W, Ci), float('nan'), device='cuda')
    K.conv_dgrad(dy_cl, wt, dx4, g, residual=res, relu_mask_bits=mbits, tf32_out=True)
    dx5 = res.clone()
    K.conv_dgrad(dy_cl, wt, dx5, g, accumulate=True, relu_mask_bits=mbits, tf32_out=True)
    torch.cuda.synchronize()
    assert torch.equal(dx4, dx2) and torch.equal(dx5, dx2)
    dw = torch.zeros((Co,) + ker + (Ci,), device='cuda')
    K.conv_wgrad(dy_cl, x_cl, dw, g)
    torch.cuda.synchronize()
    assert rel_err(dw.permute(0, 4, 1, 2, 3), wd.grad) < 2e-5


@pytest.mark.parametrize('backend', BACKENDS)
def test_stem_conv(K, backend):
    K.set_gemm_backend(backend)
    N, T, S = 2, 6, 20
    x = rnd((N, 3, T, S, S), 7)
    w = rnd((64, 3, 5, 7, 7), 8, 0.1)
    xd = x.double().requires_grad_(True)
    wd = w.double().requires_grad_(True)
    y = F.conv3d(xd, wd, None, (1, 2, 2), (2, 3, 3))
    g = K.conv_geom((N, T, S, S, 4), 64, (5, 7, 7), (1, 2, 2), (2, 3, 3))
    x4 = torch.zeros((N, T, S, S, 4))
    x4[..., :3] = to_cl(x)
    x4 = x4.cuda()
    ws = stem_pack(w).cuda()
    yd = torch.full(K.out_shape(g), float('nan'), device='cuda')
    K.conv_fwd(x4, ws, yd, g)
    torch.cuda.synchronize()
    assert rel_err(to_nc(yd), y) < 2e-5
    dy = rnd(tuple(y.shape), 9)
    y.backward(dy.double())
    dw = torch.zeros((64, 5, 7, 8, 4), device='cuda')
    mask = torch.ones((8, 4))
    mask[7, :] = 0
    mask[:, 3] = 0
    K.conv_wgrad(to_cl(dy).cuda(), x4, dw, g, col_mask=mask.reshape(32).cuda())
    torch.cuda.synchronize()
    ref = stem_pack(wd.grad)
    assert rel_err(dw, ref) < 2e-5
    assert float(dw[:, :, :, 7, :].abs().max()) == 0.0 and float(dw[..., 3].abs().max()) == 0.0


@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('N,T,S', [(2, 6, 64), (1, 3, 96), (3, 4, 32)])
def test_stem_conv_w_padded_clip_tma_path(K, backend, N, T, S):
    """conv1 on a clip whose rows are stored W-padded with zero pixels (how workspace feeds it): with Wo % 16 == 0 the
    tcgen05 engine stages the operand by TMA from the overlapping-window view (csrc/gemm_tc.cu make_tmap_stem) instead of
    16-byte cp.async gathers; results must equal the fp64 convolution for forward and weight gradient, including the
    left / right / top / bottom / temporal padding.  The layout kernel itself is checked bit for bit."""
    K.set_gemm_backend(backend)
    x = rnd((N, 3, T, S, S), 17)
    w = rnd((64, 3, 5, 7, 7), 18, 0.1)
    xd = x.double().requires_grad_(True)
    wd = w.double().requires_grad_(True)
    y = F.conv3d(xd, wd, None, (1, 2, 2), (2, 3, 3))
    g = K.conv_geom((N, T, S, S, 4), 64, (5, 7, 7), (1, 2, 2), (2, 3, 3))
    assert g.Wo % 16 == 0
    left, pitch = 3, (3 + S + 5 + 3) // 4 * 4
    buf = torch.zeros((N, T, S, pitch, 4), device='cuda')
    K.nc_to_cl(x.cuda().contiguous(), buf, N, 3, T * S * S, 4, tf32_out=True, width=S, pitch=pitch, left=left)
    torch.cuda.synchronize()
    want = torch.zeros((N, T, S, pitch, 4))
    want[:, :, :, left:left + S, :3] = to_cl(x)
    assert torch.equal(buf.cpu(), want)
    x4 = buf[:, :, :, left:left + S, :]
    assert not x4.is_contiguous()
    ws = stem_pack(w).cuda()
    yd = torch.full(K.out_shape(g), float('nan'), device='cuda')
    K.conv_fwd(x4, ws, yd, g)
    torch.cuda.synchronize()
    assert rel_err(to_nc(yd), y) < 2e-5
    dy = rnd(tuple(y.shape), 19)
    y.backward(dy.double())
    dw = torch.zeros((64, 5, 7, 8, 4), device='cuda')
    mask = torch.ones((8, 4))
    mask[7, :] = 0
    mask[:, 3] = 0
    K.conv_wgrad(to_cl(dy).cuda(), x4, dw, g, col_mask=mask.reshape(32).cuda())
    torch.cuda.synchronize()
    assert rel_err(dw, stem_pack(wd.grad)) < 2e-5
    assert float(dw[:, :, :, 7, :].abs().max()) == 0.0 and float(dw[..., 3].abs().max()) == 0.0


# -------------------------------------------------------------------------- TF32 rounding
def test_round_tf32(K):
    x = torch.randn(10007)
    y = torch.empty_like(x).cuda()
    K.round_tf32(x.cuda(), y)
    assert torch.equal(y.cpu(), tf32_round(x))


def test_truncation_vs_rounding(K):
    """Documents what the tensor core does with un-rounded fp32 operands (info for DESIGN.md)."""
    K.set_gemm_backend('tcgen05')
    g = torch.Generator().manual_seed(11)
    a = torch.randn((1, 128, 256), generator=g)
    b = torch.randn((1, 256, 128), generator=g)
    d = torch.empty((1, 128, 128), device='cuda')
    K.matmul(a.cuda(), b.cuda(), d)
    ref_exact = torch.bmm(a.double(), b.double())
    ref_rna = torch.bmm(tf32_round(a).double(), tf32_round(b).double())
    trunc = lambda t: (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)
    ref_trunc = torch.bmm(trunc(a).double(), trunc(b).double())
    print('raw fp32 operands: err vs exact %.3e, vs rna-rounded %.3e, vs truncated %.3e' % (
        rel_err(d, ref_exact), rel_err(d, ref_rna), rel_err(d, ref_trunc)))
    assert rel_err(d, ref_exact) < 5e-3


# -------------------------------------------------------------------------- streaming ops
def test_affine_nd(K):
    from oracle import ops as O
    x = torch.randn(2, 64, 3, 5, 5)
    s, b = torch.rand(64) + 0.5, torch.randn(64)
    y = torch.empty((2, 3, 5, 5, 64), device='cuda')
    K.affine_fwd(to_cl(x).cuda(), s.cuda(), b.cuda(), y)
    assert rel_err(to_nc(y), O.affine_nd(x, s, b)) < 1e-6
    K.affine_bwd(to_cl(x).cuda(), s.cuda(), y)
    assert rel_err(to_nc(y), O.affine_nd_grad(x, s)) < 1e-6


@pytest.mark.parametrize('ker,st,pd,shape', [((1, 3, 3), (1, 2, 2), (0, 1, 1), (2, 64, 4, 12, 12)),
                                             ((2, 1, 1), (2, 1, 1), (0, 0, 0), (2, 32, 8, 6, 6)),
                                             ((1, 2, 2), (1, 2, 2), (0, 0, 0), (3, 64, 4, 14, 14)),
                                             ((1, 7, 7), (1, 1, 1), (0, 0, 0), (5, 128, 1, 7, 7))])
def test_maxpool(K, ker, st, pd, shape):
    x = torch.randn(shape).double().requires_grad_(True)
    y = F.max_pool3d(x, ker, st, pd)
    dy = torch.randn(y.shape).double()
    y.backward(dy)
    N, Cc, T, H, W = shape
    g = K.conv_geom((N, T, H, W, Cc), Cc, ker, st, pd)
    xd = to_cl(x.detach().float()).cuda()
    yd = torch.empty(K.out_shape(g), device='cuda')
    arg = torch.empty(K.out_shape(g), dtype=torch.int32, device='cuda')
    K.maxpool_fwd(xd, yd, arg, g)
    assert rel_err(to_nc(yd), y) < 1e-6
    dx = torch.zeros_like(xd)
    K.maxpool_bwd(to_cl(dy.float()).cuda(), arg, dx, g)
    assert rel_err(to_nc(dx), x.grad) < 1e-5
    # gather form: no pre-zeroed buffer, same values (sums of at most a few terms, in window order)
    dxg = torch.full_like(xd, float('nan'))
    K.maxpool_bwd_gather(to_cl(dy.float()).cuda(), arg, None, dxg, g)
    assert rel_err(to_nc(dxg), x.grad) < 1e-6
    # ... with the backward of a ReLU in front of the pool folded in (mask from the pool OUTPUT) and TF32 rounding
    xr = torch.relu(x.detach()).requires_grad_(True)
    yr = F.max_pool3d(xr, ker, st, pd)
    xdr = to_cl(xr.detach().float()).cuda()
    K.maxpool_fwd(xdr, yd, arg, g)
    dxr = torch.full_like(xd, float('nan'))
    K.maxpool_bwd_gather(to_cl(dy.float()).cuda(), arg, yd, dxr, g, tf32_out=True)
    gy = to_nc(dxr).cpu()
    # reference: autograd through max-pool (ties: any winner among equal zeros is masked anyway), then relu' = (x > 0)
    yr.backward(dy)
    ref = tf32_round((xr.grad * (xr.detach() > 0)).float())
    pos = (xr.detach() > 0)
    assert torch.equal(gy[~pos], torch.zeros_like(gy[~pos]))
    assert rel_err(gy, ref) < 1e-6


@pytest.mark.parametrize('ker,shape', [((4, 1, 1), (2, 64, 4, 7, 7)), ((4, 7, 7), (2, 64, 4, 7, 7)),
                                       ((20, 1, 1), (3, 128, 20, 1, 1))])
def test_avgpool(K, ker, shape):
    x = torch.randn(shape).double().requires_grad_(True)
    y = F.avg_pool3d(x, ker, (1, 1, 1))
    dy = torch.randn(y.shape).double()
    y.backward(dy)
    N, Cc, T, H, W = shape
    g = K.conv_geom((N, T, H, W, Cc), Cc, ker, (1, 1, 1), (0, 0, 0))
    xd = to_cl(x.detach().float()).cuda()
    yd = torch.empty(K.out_shape(g), device='cuda')
    K.avgpool_fwd(xd, yd, g)
    assert rel_err(to_nc(yd), y) < 1e-5
    dx = torch.empty_like(xd)
    K.avgpool_bwd(to_cl(dy.float()).cuda(), dx, g)
    assert rel_err(to_nc(dx), x.grad) < 1e-5


def _rois(n_img, r, size, seed):
    g = torch.Generator().manual_seed(seed)
    idx = torch.randint(0, n_img, (r,), generator=g).float()
    x1 = torch.rand(r, generator=g) * size * 0.6
    y1 = torch.rand(r, generator=g) * size * 0.6
    x2 = torch.clamp(x1 + torch.rand(r, generator=g) * size * 0.6 + 2, max=size - 1)
    y2 = torch.clamp(y1 + torch.rand(r, generator=g) * size * 0.6 + 2, max=size - 1)
    rois = torch.stack([idx, x1, y1, x2, y2], 1)
    rois[0, 1:] = torch.tensor([0., 0., size - 1., size - 1.])      # full frame
    rois[1, 1:] = torch.tensor([3.3, 4.4, 3.9, 5.0])                # degenerate (< 1 cell)
    return rois


def test_roi_align_index_math_bit_exact(K):
    from oracle import roi_align_np
    for size, hw in ((224, 14), (256, 16)):
        rois = _rois(2, 40, size, 13 + size)
        pos, wts, grid = K.roi_align_table(rois.cuda(), hw, hw, 7, 7, 3, 1.0 / 16)
        pos, wts, grid = pos.cpu().numpy(), wts.cpu().numpy(), grid.cpu().numpy()
        table = roi_align_np.sample_table(rois.numpy(), hw, hw, 7, 7, 1.0 / 16, 0)
        for r, t in enumerate(table):
            assert (grid[r, 0], grid[r, 1]) == (t['grid_h'], t['grid_w'])
            gh, gw = t['grid_h'], t['grid_w']
            assert np.array_equal(pos[r, :, :, :gh, :gw], t['pos'])
            assert np.array_equal(wts[r, :, :, :gh, :gw].view(np.int32), t['w'].view(np.int32))   # bit-exact


def test_roi_align_fwd_bwd(K):
    import torchvision
    feat = torch.randn(2, 64, 14, 14).double().requires_grad_(True)
    rois = _rois(2, 9, 224, 3)
    out = torchvision.ops.roi_align(feat, rois.double(), (7, 7), 1.0 / 16, 0, False)
    dout = torch.randn(out.shape).double()
    out.backward(dout)
    fd = feat.detach().float().permute(0, 2, 3, 1).contiguous().cuda()
    od = torch.empty((9, 7, 7, 64), device='cuda')
    K.roi_align_fwd(fd, rois.cuda(), od, 1.0 / 16)
    assert rel_err(od.permute(0, 3, 1, 2), out) < 1e-5
    df = torch.zeros_like(fd)
    K.roi_align_bwd(dout.float().permute(0, 2, 3, 1).contiguous().cuda(), rois.cuda(), df, 1.0 / 16)
    assert rel_err(df.permute(0, 3, 1, 2), feat.grad) < 1e-5


@pytest.mark.parametrize('rows,cols', [(37, 784), (5, 300), (3, 3600), (64, 20)])
def test_softmax(K, rows, cols):
    x = (torch.randn(rows, cols) * 3).double().requires_grad_(True)
    p = torch.softmax(x * 0.25, dim=1)
    dp = torch.randn(rows, cols).double()
    p.backward(dp)
    pd = torch.empty((rows, cols), device='cuda')
    K.softmax_fwd(x.detach().float().cuda(), pd, 0.25)
    assert rel_err(pd, p) < 1e-5
    dx = torch.empty_like(pd)
    K.softmax_bwd(pd, dp.float().cuda(), dx, 0.25)
    assert rel_err(dx, x.grad) < 1e-4
    dxr = torch.empty_like(pd)
    K.softmax_bwd(pd, dp.float().cuda(), dxr, 0.25, tf32_out=True)      # the same values, stored TF32-rounded
    want = torch.empty_like(dx)
    K.round_tf32(dx, want)
    torch.cuda.synchronize()
    assert torch.equal(dxr, want)


def test_layernorm(K):
    from oracle import ops as O
    x = torch.randn(7, 512).double().requires_grad_(True)
    y, mean, std = O.layer_norm_axis1(x)
    dy = torch.randn(7, 512).double()
    y.backward(dy)
    yd = torch.empty((7, 512), device='cuda')
    md, sd = torch.empty(7, device='cuda'), torch.empty(7, device='cuda')
    K.layernorm_fwd(x.detach().float().cuda(), yd, md, sd, 512)
    assert rel_err(yd, y) < 1e-5 and rel_err(sd, std.view(-1)) < 1e-5 and rel_err(md, mean.view(-1)) < 1e-4
    dx = torch.empty_like(yd)
    K.layernorm_bwd(dy.float().cuda(), yd, sd, dx, 512)
    assert rel_err(dx, x.grad) < 1e-4


def test_elementwise_and_layout(K):
    x = torch.randn(1003)
    y = torch.randn(1003)
    o = torch.empty(1003, device='cuda')
    K.relu_fwd(x.cuda(), o)
    assert torch.equal(o.cpu(), torch.relu(x))
    K.relu_bwd(x.cuda(), y.cuda(), o)
    assert torch.equal(o.cpu(), x * (y > 0))
    K.axpby(x.cuda(), 2.0, y.cuda(), -0.5, o)
    assert rel_err(o, 2 * x - 0.5 * y) < 1e-6
    K.fill(o, 3.0)
    assert float(o.min()) == 3.0 and float(o.max()) == 3.0
    K.sigmoid_fwd(x.cuda(), o)
    assert rel_err(o, torch.sigmoid(x)) < 1e-6
    # fused gradient finish: sum of two contributions + ReLU backward + TF32 rounding, bit-exact vs the two-pass form
    for n in (1003, 4096):
        a, b, m = torch.randn(n), torch.randn(n), torch.randn(n)
        want = tf32_round(a + b) * (m > 0)
        ad = a.cuda()
        K.add_relu_bwd_tf32(ad, b.cuda(), m.cuda(), ad)          # in place on a
        assert torch.equal(ad.cpu(), want)
        od = torch.empty(n, device='cuda')
        K.add_relu_bwd_tf32(a.cuda(), b.cuda(), None, od)
        assert torch.equal(od.cpu(), tf32_round(a + b))
    # layouts
    t = torch.randn(2, 3, 4, 5, 6)
    cl = torch.empty((2, 4, 5, 6, 4), device='cuda')
    K.nc_to_cl(t.cuda(), cl, 2, 3, 4 * 5 * 6, 4)
    assert torch.equal(cl[..., :3].cpu(), to_cl(t)) and float(cl[..., 3].abs().max()) == 0
    # clip feeding: the vectorised C<=4 path (inner % 4 == 0), with and without the fused TF32 rounding, the generic
    # path for a ragged inner extent (7*5*3 = 105), and a 1-plane / 4-plane input
    for shape in [(2, 3, 8, 16, 16), (1, 3, 7, 5, 3), (2, 1, 4, 4, 4), (3, 4, 2, 6, 6)]:
        tc_ = torch.randn(shape)
        n_, c_, inner_ = shape[0], shape[1], shape[2] * shape[3] * shape[4]
        for rnd_ in (False, True):
            o = torch.full((n_,) + shape[2:] + (4,), float('nan'), device='cuda')
            K.nc_to_cl(tc_.cuda(), o, n_, c_, inner_, 4, tf32_out=rnd_)
            want = to_cl(tc_)
            assert torch.equal(o[..., :c_].cpu(), tf32_round(want) if rnd_ else want), (shape, rnd_)
            assert c_ == 4 or float(o[..., c_:].abs().max()) == 0
    t2 = torch.randn(3, 70, 2, 3, 3)
    cl2 = torch.empty((3, 2, 3, 3, 70), device='cuda')
    K.nc_to_cl(t2.cuda(), cl2, 3, 70, 18)
    assert torch.equal(cl2.cpu(), to_cl(t2))
    back = torch.empty((3, 70, 2, 3, 3), device='cuda')
    K.cl_to_nc(cl2, back, 3, 70, 18)
    assert torch.equal(back.cpu(), t2)
    # copy2d / dropout
    src = torch.randn(5, 7).cuda()
    dst = torch.zeros(5, 20).cuda()
    K.copy2d(src, 7, dst, 20, 5, 7, dst_off=8)
    assert torch.equal(dst[:, 8:15], src) and float(dst[:, :8].abs().max()) == 0
    big = torch.ones(100000).cuda()
    out = torch.empty_like(big)
    K.dropout(big, out, 0.3, 1234, 0)
    keep = float((out > 0).float().mean())
    assert abs(keep - 0.7) < 0.01 and abs(float(out.max()) - 1 / 0.7) < 1e-5
    out2 = torch.empty_like(big)
    K.dropout(big, out2, 0.3, 1234, 0)
    assert torch.equal(out, out2)
    step = torch.zeros(1, dtype=torch.int64, device='cuda')
    K.dropout(big, out2, 0.3, 1234, 0, step)
    assert torch.equal(out, out2)                    # step 0 == no step
    step.fill_(5)
    K.dropout(big, out2, 0.3, 1234, 0, step)
    assert not torch.equal(out, out2) and abs(float((out2 > 0).float().mean()) - 0.7) < 0.01


def test_losses_and_sgd(K):
    from oracle import ops as O
    x = (torch.randn(6, 80) * 2).double().requires_grad_(True)
    t = (torch.rand(6, 80) < 0.1).int()
    t[0, :5] = -1
    loss = O.sigmoid_cross_entropy_loss(x, t, 0.125)
    loss.backward()
    ld = torch.empty(1, device='cuda')
    K.sigmoid_ce_fwd(x.detach().float().cuda(), t.cuda(), ld, 0.125)
    assert rel_err(ld, loss.view(1)) < 1e-5
    dx = torch.empty((6, 80), device='cuda')
    K.sigmoid_ce_bwd(x.detach().float().cuda(), t.cuda(), None, dx, 0.125)
    assert rel_err(dx, x.grad) < 1e-5
    x2 = torch.randn(5, 157).double().requires_grad_(True)
    lab = torch.randint(0, 157, (5,)).int()
    prob, l2 = O.softmax_with_loss(x2, lab, 0.5)
    l2.backward()
    pd, l2d = torch.empty((5, 157), device='cuda'), torch.empty(1, device='cuda')
    K.softmax_ce_fwd(x2.detach().float().cuda(), lab.cuda(), pd, l2d, 0.5)
    assert rel_err(pd, prob) < 1e-5 and rel_err(l2d, l2.view(1)) < 1e-5
    dx2 = torch.empty_like(pd)
    K.softmax_ce_bwd(pd, lab.cuda(), dx2, 0.5)
    assert rel_err(dx2, x2.grad) < 1e-5
    p, g, m = torch.randn(1001), torch.randn(1001), torch.randn(1001)
    pr, mr = O.nesterov_update(p.double(), g.double(), m.double(), 0.04, 0.9, 1e-3)
    pd_, gd_, md_ = p.cuda(), g.cuda(), m.cuda()
    pt = torch.empty_like(pd_)
    K.sgd_nesterov(pd_, gd_, md_, torch.tensor([0.04], device='cuda'), 0.9, 1e-3, True, pt)
    assert rel_err(pd_, pr) < 1e-6 and rel_err(md_, mr) < 1e-6
    assert torch.equal(pt.cpu(), tf32_round(pd_.cpu()))


@pytest.mark.parametrize('rows,cols', [(1200, 512), (25088, 256), (3, 80), (70000, 64)] +
                         [(r, c) for r in (1, 63, 64, 65) for c in (1, 157)])
def test_colsum(K, rows, cols):
    """Dense and strided (a column block of a matrix twice as wide, ld = 2 cols) inputs, one row slab (rows <= 64)
    and several (partial sums added in slab order); stored, then added into a random out."""
    wide = torch.randn(rows, 2 * cols)
    for x, ld in ((wide[:, :cols].contiguous(), cols), (wide[:, cols:], 2 * cols)):
        s = x.double().sum(0)
        xd = x.contiguous().cuda() if ld == cols else wide.cuda()[:, cols:]
        out = torch.full((cols,), 7.0, device='cuda')
        K.colsum(xd, ld, out, rows, cols, accumulate=False)
        assert rel_err(out, s) < 1e-5, ld
        out0 = torch.randn(cols) * float(s.abs().max())
        out = out0.cuda()
        K.colsum(xd, ld, out, rows, cols, accumulate=True)
        assert rel_err(out.cpu().double() - out0.double(), s) < 1e-5, ld


def test_weight_transpose_multi_matches_single(K):
    """One launch for all dgrad weight operands of a step == the per-conv kernel."""
    shapes = [(64, 1, 1, 1, 64), (96, 3, 1, 1, 32), (40, 1, 3, 3, 72), (512, 1, 1, 1, 2048)]
    jobs, refs = [], []
    for i, shp in enumerate(shapes):
        w = torch.randn(shp, device='cuda')
        sc = (torch.rand(shp[0], device='cuda') + 0.5) if i % 2 == 0 else None
        taps = shp[1] * shp[2] * shp[3]
        wt = torch.full((shp[4], taps, shp[0]), float('nan'), device='cuda')
        ref = torch.empty_like(wt)
        K.weight_transpose(w, ref, sc)
        jobs.append((w, wt, sc))
        refs.append(ref)
    cache = {}
    K.weight_transpose_multi(jobs, cache)
    K.weight_transpose_multi(jobs, cache)          # second call reuses the device job table
    torch.cuda.synchronize()
    for (w, wt, sc), ref in zip(jobs, refs):
        assert torch.equal(wt, ref)


# -------------------------------------------------------------------------- raw-bank kernels (csrc/fbo.cu)
@pytest.mark.parametrize('R,Lb,D', [(1, 1, 2048), (3, 7, 2048), (4, 300, 2048), (2, 301, 1024), (5, 60, 4096),
                                     (37, 120, 2048), (3, 3600, 2048)])
def test_fbo_bank_scan(K, R, Lb, D):
    """One pass over the raw bank: scores q.b_j, softmax over the L rows, weighted row sum -- against fp64; ragged
    tails (L not a multiple of the 8-row tile or of the split), one-row banks, zero-padded rows, every supported D."""
    g = torch.Generator().manual_seed(R * 1000 + Lb)
    bank = torch.randn((R, Lb, D), generator=g) * 0.5
    bank[:, Lb - Lb // 4:] = 0.0                        # the reference zero-pads short windows (ava.py:310-321)
    q = torch.randn((R, D), generator=g) * 0.2
    sc = 512 ** -0.5
    p = torch.softmax(torch.einsum('rld,rd->rl', bank.double(), q.double()) * sc, dim=1)
    ref = torch.einsum('rl,rld->rd', p, bank.double())
    out = torch.full((R, D), float('nan'), device='cuda')
    prob = torch.full((R, Lb), float('nan'), device='cuda')
    K.fbo_bank_scan(bank.cuda(), q.cuda(), out, sc, prob=prob)
    torch.cuda.synchronize()
    assert rel_err(prob, p) < 1e-5 and rel_err(out, ref) < 1e-5
    out2 = torch.empty_like(out)
    K.fbo_bank_scan(bank.cuda(), q.cuda(), out2, sc, prob=None, tf32_out=True)
    assert torch.equal(out2.cpu(), tf32_round(out.cpu()))


@pytest.mark.parametrize('R,Lb,D', [(1, 1, 2048), (3, 7, 2048), (4, 300, 2048), (5, 61, 4096), (37, 120, 2048),
                                     (2, 3600, 2048)])
def test_fbo_bank_scan_bf16_bank(K, R, Lb, D):
    """The same pass over a bank STORED as bf16 (vlfb_fbo_bank_scan_dt, VLFB_DT_BF16): the cast kernel rounds to nearest
    even bit-exactly like torch, and the scan of the bf16 bank equals the fp64 evaluation on the rounded values (the
    arithmetic stays fp32), ragged tails and zero-padded rows included."""
    g = torch.Generator().manual_seed(R * 1000 + Lb + 1)
    bank = torch.randn((R, Lb, D), generator=g) * 0.5
    bank[:, Lb - Lb // 4:] = 0.0
    q = torch.randn((R, D), generator=g) * 0.2
    b16 = torch.empty((R, Lb, D), dtype=torch.bfloat16, device='cuda')
    K.cast_bf16(bank.cuda().view(-1), b16.view(-1))
    assert torch.equal(b16.cpu(), bank.to(torch.bfloat16))
    sc = 512 ** -0.5
    bd = b16.cpu().double()
    p = torch.softmax(torch.einsum('rld,rd->rl', bd, q.double()) * sc, dim=1)
    ref = torch.einsum('rl,rld->rd', p, bd)
    out = torch.full((R, D), float('nan'), device='cuda')
    prob = torch.full((R, Lb), float('nan'), device='cuda')
    K.fbo_bank_scan(b16, q.cuda(), out, sc, prob=prob)
    torch.cuda.synchronize()
    assert rel_err(prob, p) < 1e-5 and rel_err(out, ref) < 1e-5
    lib = K.L.load()
    s = lib.vlfb_fbo_bank_scan_splits_dt(R, Lb, D, 1)
    assert s >= 1 and lib.vlfb_fbo_bank_scan_workspace_dt(R, Lb, D, 1) == (R * s * D + R * s * 2) * 4
    assert lib.vlfb_fbo_bank_scan_splits_dt(R, Lb, 1024, 1) == 0          # bf16 rows: 2048 / 4096 features only


def test_fbo_bank_scan_peaked_softmax_and_split_table(K):
    """Scores far apart (one row dominates): the online softmax must not overflow / lose the winner across CTA splits;
    and the split chooser keeps every CTA non-empty."""
    from vlfb import libvlfb as L
    lib = L.load()
    for R, Lb in [(1, 1), (4, 300), (256, 3600), (64, 60), (3, 9), (1000, 17)]:
        s = lib.vlfb_fbo_bank_scan_splits(R, Lb, 2048)
        per = (Lb + s - 1) // s
        assert s >= 1 and (s - 1) * per < Lb
    assert lib.vlfb_fbo_bank_scan_splits(4, 300, 1000) == 0
    R, Lb, D = 2, 300, 2048
    bank = torch.randn(R, Lb, D)
    q = torch.zeros(R, D)
    q[0] = bank[0, 123] * 5.0          # score(123) ~ 5 * 2048: every other row underflows to exactly 0
    q[1] = -bank[1, 299] * 5.0         # the last row gets the most NEGATIVE score
    out = torch.empty((R, D), device='cuda')
    prob = torch.empty((R, Lb), device='cuda')
    K.fbo_bank_scan(bank.cuda(), q.cuda(), out, 1.0, prob=prob)
    p = torch.softmax(torch.einsum('rld,rd->rl', bank.double(), q.double()), dim=1)
    assert torch.isfinite(out).all() and rel_err(prob, p) < 1e-5
    assert rel_err(out, torch.einsum('rl,rld->rd', p, bank.double())) < 1e-5
    assert abs(float(prob[0, 123]) - 1.0) < 1e-6


def test_fbo_bank_scan_rejects_bad_arguments(K):
    from vlfb import libvlfb as L
    bank, q, out = torch.zeros((2, 8, 512), device='cuda'), torch.zeros((2, 512), device='cuda'), torch.zeros((2, 512), device='cuda')
    with pytest.raises(L.VlfbError):
        K.fbo_bank_scan(bank, q, out, 1.0)
    lib = L.load()
    b2 = torch.zeros((2, 8, 2048), device='cuda')
    rc = lib.vlfb_fbo_bank_scan(b2.data_ptr(), b2.data_ptr(), 1.0, b2.data_ptr(), None, 2, 8, 2048, 0, None, 0, None)
    assert rc == -4 and b'workspace' in lib.vlfb_last_error()


@pytest.mark.parametrize('rows,n,D', [(1000, 600, 2048), (17, 5, 64), (3, 0, 2048), (50000, 4800, 2048)])
def test_lfb_gather_is_bit_exact(K, rows, n, D):
    g = torch.Generator().manual_seed(rows + n)
    bank = torch.randn((rows, D), generator=g)
    idx = torch.randint(-1, rows, (n,), generator=g, dtype=torch.int32)
    if n > 2:
        idx[0], idx[-1] = -1, rows - 1
    ref = torch.zeros((n, D))
    ok = idx >= 0
    ref[ok] = bank[idx[ok].long()]
    out = torch.full((n, D), float('nan'), device='cuda')
    K.lfb_gather(bank.cuda(), idx.cuda(), out)
    assert torch.equal(out.cpu(), ref)
    K.lfb_gather(bank.cuda(), idx.cuda(), out, tf32_out=True)
    assert torch.equal(out.cpu(), tf32_round(ref))


# -------------------------------------------------------------------------- tiling / schedule variants
# vlfb_gemm_params_t.{tile_n, pair, stream_k}: 256-row tiles on CTA pairs (tcgen05 cta_group::2), stream-K chunk
# ranges with the workspace fix-up, forced tile widths.  Every variant must reproduce the fp64 reference at the
# production shapes of res4 / res5 / the non-local blocks (M = 6272 = 2 clips x 16 x 14 x 14).
VARIANTS = [dict(pair=-1, stream_k=-1), dict(pair=1, stream_k=-1), dict(pair=-1, stream_k=1), dict(pair=1, stream_k=1),
            dict(pair=-1, stream_k=-1, tile_n=192), dict(pair=1, stream_k=1, tile_n=128), dict()]


def _with_opts(K, opts):
    K.GEMM_OPTS.update(dict(tile_n=0, pair=0, stream_k=0))
    K.GEMM_OPTS.update(opts)


def _conv_ref_gpu(x_cl, w_cl, st, pd, dil):
    """fp64 reference on the GPU (cuDNN / native double convolution: independent of libvlfb)."""
    x = x_cl.permute(0, 4, 1, 2, 3).double()
    w = w_cl.permute(0, 4, 1, 2, 3).double()
    return F.conv3d(x, w, None, st, pd, dil).permute(0, 2, 3, 4, 1).contiguous()


PROD_CONVS = [
    # Ci, Co, kernel, pads, dilation, residual        (N, T, H, W) = (2, 16, 14, 14): M = 6272
    (512, 512, (1, 3, 3), (0, 2, 2), (1, 2, 2), False),      # res5 branch2b   K = 4608
    (2048, 512, (3, 1, 1), (1, 0, 0), (1, 1, 1), False),     # res5 branch2a   K = 6144
    (256, 256, (1, 3, 3), (0, 1, 1), (1, 1, 1), False),      # res4 branch2b   K = 2304
    (1024, 256, (3, 1, 1), (1, 0, 0), (1, 1, 1), False),     # res4 branch2a   K = 3072
    (256, 1024, (1, 1, 1), (0, 0, 0), (1, 1, 1), True),      # res4 branch2c + residual + ReLU
    (512, 2048, (1, 1, 1), (0, 0, 0), (1, 1, 1), True),      # res5 branch2c
]


@pytest.mark.parametrize('case', range(len(PROD_CONVS)))
def test_production_conv_shapes_all_tiling_variants(K, case):
    K.set_gemm_backend('tcgen05')
    Ci, Co, ker, pd, dil, use_res = PROD_CONVS[case]
    g = K.conv_geom((2, 16, 14, 14, Ci), Co, ker, (1, 1, 1), pd, dil)
    x = rnd((2, 16, 14, 14, Ci), 40 + case).cuda()
    w = rnd((Co,) + tuple(ker) + (Ci,), 50 + case, 0.05).cuda()
    s, b = (torch.rand(Co) + 0.5).cuda(), torch.randn(Co).cuda()
    res = rnd(K.out_shape(g), 60 + case).cuda() if use_res else None
    dy = rnd(K.out_shape(g), 70 + case).cuda()
    y_ref = _conv_ref_gpu(x, w, (1, 1, 1), pd, dil)
    out_ref = y_ref * s.double() + b.double()
    if use_res:
        out_ref = out_ref + res.double()
    out_ref = torch.relu(out_ref)
    taps = ker[0] * ker[1] * ker[2]
    wt = torch.empty((Ci, taps, Co), device='cuda')
    K.weight_transpose(w, wt)
    # dgrad reference: conv_transpose == autograd of the fp64 conv
    xd = x.permute(0, 4, 1, 2, 3).double().requires_grad_(True)
    wd = w.permute(0, 4, 1, 2, 3).double().requires_grad_(True)
    yy = F.conv3d(xd, wd, None, (1, 1, 1), pd, dil)
    yy.backward(dy.permute(0, 4, 1, 2, 3).double())
    dx_ref = xd.grad.permute(0, 2, 3, 4, 1)
    dw_ref = wd.grad.permute(0, 2, 3, 4, 1) * s.double().view(-1, 1, 1, 1, 1)
    dw0 = torch.randn(tuple(dw_ref.shape), generator=torch.Generator().manual_seed(80 + case)) * float(dw_ref.abs().max())
    xbits = pack_sign_bits(x)
    try:
        for opts in VARIANTS:
            _with_opts(K, opts)
            y = torch.full(K.out_shape(g), float('nan'), device='cuda')
            ybits = torch.zeros((y.numel() // 32,), dtype=torch.int32, device='cuda')
            K.conv_fwd(x, w, y, g, scale=s, bias=b, residual=res, relu=True, relu_bits=ybits)
            dx = torch.full((2, 16, 14, 14, Ci), float('nan'), device='cuda')
            K.conv_dgrad(dy, wt, dx, g)
            # finishing dgrad: + residual, ReLU mask as sign bits, TF32 rounding (the epilogue of the training step)
            dxf = torch.full((2, 16, 14, 14, Ci), float('nan'), device='cuda')
            K.conv_dgrad(dy, wt, dxf, g, residual=x, relu_mask_bits=xbits, tf32_out=True)
            dw = dw0.cuda()                   # accumulated: dw = pattern + row_scale * grad
            K.conv_wgrad(dy, x, dw, g, row_scale=s)
            torch.cuda.synchronize()
            assert rel_err(y, out_ref) < 2e-5, ('fwd', opts)
            assert torch.equal(ybits, pack_sign_bits(y)), ('fwd sign bits', opts)
            assert rel_err(dx, dx_ref) < 2e-5, ('dgrad', opts)
            assert rel_err(dxf, (dx_ref + x.double()) * (x > 0)) < 6e-4, ('finishing dgrad', opts)
            assert (dxf[x <= 0] == 0).all() and (dxf.view(torch.int32) & 0x1FFF).eq(0).all()
            assert rel_err(dw.double().cpu() - dw0.double(), dw_ref) < 2e-5, ('wgrad', opts)
            # the counters of the stream-K workspace are zero again after every launch
            assert int(K.gemm_workspace(x.device)[:16384].view(torch.int32).abs().sum()) == 0, opts
    finally:
        _with_opts(K, {})


@pytest.mark.parametrize('B,M,N,K_,ta,tb', [(2, 3136, 784, 512, 1, 0),      # NL4 affinity theta^T phi (MN-major A)
                                            (2, 512, 3136, 784, 0, 1),      # NL4 y = g p^T
                                            (8, 3136, 784, 256, 1, 0),      # NL3 (grouped) affinity
                                            (1, 6272, 1024, 512, 0, 1),     # NL4 out projection as a matmul
                                            (1, 300, 520, 2048, 0, 1)])     # ragged M / N
def test_production_matmul_shapes_all_tiling_variants(K, B, M, N, K_, ta, tb):
    K.set_gemm_backend('tcgen05')
    a = rnd((B, K_, M) if ta else (B, M, K_), 81).cuda()
    b = rnd((B, N, K_) if tb else (B, K_, N), 82).cuda()
    A = a.transpose(1, 2) if ta else a
    Bm = b.transpose(1, 2) if tb else b
    bias = torch.randn(N).cuda()
    ref = torch.bmm(A.double(), Bm.double()) + bias.double()
    try:
        for opts in VARIANTS:
            _with_opts(K, opts)
            d = torch.full((B, M, N), float('nan'), device='cuda')
            K.matmul(A, Bm, d, bias=bias)
            torch.cuda.synchronize()
            assert rel_err(d, ref) < 2e-5, opts
            K.matmul(A, Bm, d, accumulate=True)
            torch.cuda.synchronize()
            assert rel_err(d, 2 * ref - bias.double()) < 2e-5, opts
    finally:
        _with_opts(K, {})


def test_stream_k_results_are_deterministic(K):
    """The fix-up sums the pieces of a shared tile in piece order, whoever arrives last: two runs are bit-identical."""
    K.set_gemm_backend('tcgen05')
    g = K.conv_geom((2, 16, 14, 14, 512), 512, (1, 3, 3), (1, 1, 1), (0, 2, 2), (1, 2, 2))
    x, w = rnd((2, 16, 14, 14, 512), 91).cuda(), rnd((512, 1, 3, 3, 512), 92, 0.05).cuda()
    try:
        _with_opts(K, dict(pair=1, stream_k=1))
        outs = []
        for _ in range(3):
            y = torch.empty(K.out_shape(g), device='cuda')
            K.conv_fwd(x, w, y, g, relu=True, tf32_out=True)
            torch.cuda.synchronize()
            outs.append(y.clone())
        assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    finally:
        _with_opts(K, {})



def test_gradient_reductions_are_deterministic(K):
    """Every reduction of the training step's backward that many CTAs share -- a weight gradient over a long K (the
    library picks the split), a skinny long-K matmul, bias-gradient column sums and the RoIAlign backward -- gives
    bit-identical results run after run: none of them depends on the order in which blocks finish."""
    K.set_gemm_backend('tcgen05')
    g = K.conv_geom((2, 8, 28, 28, 256), 256, (1, 3, 3), (1, 1, 1), (0, 1, 1))
    x = rnd((2, 8, 28, 28, 256), 93).cuda()
    dy = rnd(K.out_shape(g), 94).cuda()
    a, b = rnd((1, 4, 2560), 95).cuda(), rnd((1, 2560, 80), 96).cuda()
    rows = rnd((50000, 80), 97).cuda()
    feat_g = rnd((4, 7, 7, 256), 98).cuda()
    rois = torch.tensor([[0, 0., 0., 223., 223.], [1, 10.5, 20.25, 100.75, 180.5], [0, 3.3, 4.4, 30.9, 25.0],
                         [1, 111., 7., 223., 60.]], device='cuda')
    outs = []
    for _ in range(3):
        dw = torch.zeros((256, 1, 3, 3, 256), device='cuda')
        K.conv_wgrad(dy, x, dw, g)
        d = torch.empty((1, 4, 80), device='cuda')
        K.matmul(a, b, d)
        cs = torch.empty(80, device='cuda')
        K.colsum(rows, 80, cs, 50000, 80, accumulate=False)
        df = torch.zeros((2, 14, 14, 256), device='cuda')
        K.roi_align_bwd(feat_g, rois, df, 1.0 / 16)
        torch.cuda.synchronize()
        outs.append((dw, d, cs, df))
    for o in outs[1:]:
        for u, v in zip(outs[0], o):
            assert torch.equal(u, v)
    assert outs[0][3].abs().sum() > 0 and outs[0][0].abs().sum() > 0

# -------------------------------------------------------------------------- training-mode FBO-NL stack (one launch)
def _fbo_ref(a0, bp, Ws, scale, pre_act_ln, eps=1e-5):
    """As-written NLLayers / NLCore (lfb_helper.py:170-292) in fp64 with autograd: phi and g ARE formed here."""
    A = a0
    outs = []
    for W in Ws:
        theta = A @ W['w_theta'].t() + W['b_theta']                       # (R, d)
        phi = bp @ W['w_phi'].t() + W['b_phi']                             # (R, L, d)
        g = bp @ W['w_g'].t() + W['b_g']
        aff = torch.einsum('rd,rld->rl', theta, phi) * scale
        p = torch.softmax(aff, dim=1)
        t = torch.einsum('rl,rld->rd', p, g)
        x = F.layer_norm(t, (t.shape[1],), eps=eps) if pre_act_ln else t
        out = torch.relu(x) @ W['w_out'].t() + W['b_out']
        A = A + out
        outs.append(dict(theta=theta, prob=p, t=t, out=out, a_out=A))
    return A, outs


@pytest.mark.parametrize('R,L,dA,d,dB,layers,ln', [(4, 300, 512, 512, 512, 2, True), (3, 37, 512, 512, 512, 3, True),
                                                    (5, 60, 2048, 512, 512, 2, True), (2, 120, 512, 512, 512, 1, False)])
def test_fbo_nl_stack_fwd_bwd(K, R, L, dA, d, dB, layers, ln):
    """vlfb_fbo_nl_fwd / _bwd (phi and g folded onto the projected bank) against the as-written graph in fp64:
    every saved activation, the input / bank gradients and all weight / bias gradients, incl. zero-padded bank rows
    (they still receive softmax mass, lfb_helper.py NTC_to_NCT11 note) and a b_phi whose gradient is exactly 0."""
    g = torch.Generator().manual_seed(7)
    rn = lambda *s, sc=1.0: (torch.randn(*s, generator=g) * sc)
    a0 = rn(R, dA)
    bp = rn(R, L, dB, sc=0.7)
    bp[:, L - L // 4:] = 0.0
    scale = d ** -0.5
    Ws = [dict(w_theta=rn(d, dA, sc=0.05), b_theta=rn(d, sc=0.1), w_phi=rn(d, dB, sc=0.08), b_phi=rn(d, sc=0.1),
               w_g=rn(d, dB, sc=0.05), b_g=rn(d, sc=0.1), w_out=rn(dA, d, sc=0.05), b_out=rn(dA, sc=0.1))
          for _ in range(layers)]
    a64 = a0.double().requires_grad_(True)
    b64 = bp.double().requires_grad_(True)
    W64 = [dict((k, v.double().requires_grad_(True)) for k, v in W.items()) for W in Ws]
    A_ref, outs = _fbo_ref(a64, b64, W64, scale, ln)
    dlast = rn(R, dA)
    (A_ref * dlast.double()).sum().backward()

    dev = lambda t: t.float().cuda().contiguous()
    lay = []
    for W in Ws:
        ld = dict((k, dev(v)) for k, v in W.items())
        for k, v in W.items():
            ld['g' + k] = torch.full(v.shape, 0.25, device='cuda')             # accumulated into: starts non-zero
        ld.update(theta=torch.empty(R, d, device='cuda'), prob=torch.empty(R, L, device='cuda'),
                  s=torch.empty(R, dB, device='cuda'), t=torch.empty(R, d, device='cuda'),
                  xhat=torch.empty(R, d, device='cuda'), ln_mean=torch.empty(R, device='cuda'),
                  ln_std=torch.empty(R, device='cuda'), out=torch.empty(R, dA, device='cuda'),
                  a_out=torch.empty(R, dA, device='cuda'))
        lay.append(ld)
    cfgd = dict(R=R, L=L, dA=dA, d=d, dB=dB, scale=scale, pre_act_ln=ln)
    K.fbo_nl_fwd(cfgd, lay, dev(a0), dev(bp))
    torch.cuda.synchronize()
    for ld, o in zip(lay, outs):
        for k in ('theta', 'prob', 't', 'out', 'a_out'):
            assert rel_err(ld[k], o[k]) < 2e-5, k
    da0 = torch.full((R, dA), float('nan'), device='cuda')
    dbp = torch.full((R, L, dB), float('nan'), device='cuda')
    K.fbo_nl_bwd(cfgd, lay, dev(a0), dev(bp), dev(dlast), da0, dbp)
    torch.cuda.synchronize()
    assert rel_err(da0, a64.grad) < 5e-5
    assert rel_err(dbp, b64.grad) < 5e-5
    for ld, W in zip(lay, W64):
        for k, v in W.items():
            got = ld['g' + k].cpu().double() - 0.25
            if k == 'b_phi':                                                   # exactly zero in exact arithmetic
                assert float(got.abs().max()) < 1e-5 and float(v.grad.abs().max()) < 1e-9
            else:
                assert rel_err(got, v.grad) < 1e-4, k


def test_fbo_nl_stack_dropout_is_an_unbiased_philox_mask(K):
    """drop_ratio > 0: each element of a layer's output is kept with probability 1 - ratio and scaled by 1 / (1 - ratio);
    the same (seed, offset) gives the same mask forward and backward (da0 of a pure-residual probe)."""
    R, L, dA = 8, 20, 512
    ld = dict(w_theta=torch.zeros(512, dA, device='cuda'), b_theta=torch.zeros(512, device='cuda'),
              w_phi=torch.zeros(512, 512, device='cuda'), b_phi=None, w_g=torch.zeros(512, 512, device='cuda'),
              b_g=torch.ones(512, device='cuda'), w_out=torch.zeros(dA, 512, device='cuda'),
              b_out=torch.ones(dA, device='cuda'), theta=torch.empty(R, 512, device='cuda'),
              prob=torch.empty(R, L, device='cuda'), s=torch.empty(R, 512, device='cuda'),
              t=torch.empty(R, 512, device='cuda'), xhat=torch.empty(R, 512, device='cuda'),
              ln_mean=torch.empty(R, device='cuda'), ln_std=torch.empty(R, device='cuda'),
              out=torch.empty(R, dA, device='cuda'), a_out=torch.empty(R, dA, device='cuda'), drop_offset=12345)
    a0 = torch.zeros(R, dA, device='cuda')
    bp = torch.randn(R, L, 512, device='cuda')
    cfgd = dict(R=R, L=L, dA=dA, d=512, dB=512, scale=1.0, pre_act_ln=False, drop_ratio=0.2, seed=99)
    K.fbo_nl_fwd(cfgd, [ld], a0, bp)
    torch.cuda.synchronize()
    a = ld['a_out'].cpu()                                   # out == 1 everywhere -> a_out is the scaled keep mask
    vals = set(np.round(a.unique().numpy(), 5).tolist())
    assert vals == {0.0, 1.25}
    assert abs(float((a > 0).float().mean()) - 0.8) < 0.02
    x = torch.empty(R * dA, device='cuda')
    K.dropout(torch.ones(R * dA, device='cuda'), x, 0.2, 99, 12345)
    assert torch.equal(x.view(R, dA).cpu(), a), 'same generator as vlfb_dropout_fwd'
