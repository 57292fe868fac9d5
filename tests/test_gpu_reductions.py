"""The reductions of the training step's backward that many CTAs share, tested at their edges: the RoIAlign backward
(a gather), the accumulating GEMM (whole tiles or stream-K pieces summed in a fixed order), and colsum (slab partial
sums).  Each is compared with an fp64 reference, and each must give the same bits run after run -- as must a whole
training step.

RoIAlign is linear in the feature map, so its reference is one dense fp64 matrix A[(r, ph, pw), (n, y, x)] built from
the sample table of oracle/roi_align_np.py: forward = A @ feat, backward = A^T @ dout.  A itself is checked against
torchvision's roi_align (aligned=False) in float64, on the CPU."""
import ctypes

import numpy as np
import pytest
import torch

import harness as H
from util import rel_err, stem_pack, tf32_round

gpu = pytest.mark.gpu


@pytest.fixture(scope='module')
def K():
    from vlfb import kernels
    assert torch.cuda.is_available()
    yield kernels
    kernels.set_gemm_backend('tcgen05')


def rnd(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return tf32_round(torch.randn(shape, generator=g) * scale)


def bits(t):
    return t.detach().cpu().contiguous().view(torch.int32)


# -------------------------------------------------------------------------- RoIAlign
def _box(n, x1, y1, x2, y2):
    return [float(n), x1, y1, x2, y2]


def _random_rois(imgs, r, size, seed, lo=0.0, span=0.6, min_w=2.0):
    g = torch.Generator().manual_seed(seed)
    idx = torch.tensor(imgs)[torch.randint(0, len(imgs), (r,), generator=g)].float()
    x1 = torch.rand(r, generator=g) * size * span + lo
    y1 = torch.rand(r, generator=g) * size * span + lo
    x2 = x1 + torch.rand(r, generator=g) * size * span + min_w
    y2 = y1 + torch.rand(r, generator=g) * size * span + min_w
    return torch.stack([idx, x1, y1, x2, y2], 1)


# name -> (N, H, W, C, PH, PW, spatial_scale, sampling_ratio, rois [R, 5])
def _roi_cases():
    c = {}
    # past every border: samples in the clamped bands (-1, 0] and [L-1, L], and beyond them (dropped)
    c['borders'] = (2, 14, 14, 36, 7, 7, 1 / 16, 0, [
        _box(0, -40, -30, 100, 90), _box(1, 150, 160, 260, 250), _box(0, -20, 100, 240, 130),
        _box(1, -24, -8, 8, 232), _box(0, 200, -16, 236, 40), _box(1, -30, -30, 250, 250)])
    # entirely outside the map: zero output, no gradient; next to a RoI inside so that the image is not empty
    c['outside'] = (2, 14, 14, 36, 7, 7, 1 / 16, 0, [
        _box(0, 300, 300, 400, 400), _box(1, -100, -100, -40, -40), _box(1, 20, 30, 120, 90),
        _box(0, -200, 50, -30, 120)])
    # degenerate: x2 < x1 / y2 < y1 (the size is clamped to one cell) and boxes under one cell
    c['degenerate'] = (2, 14, 14, 36, 7, 7, 1 / 16, 0, [
        _box(0, 50, 60, 30, 40), _box(1, 33.3, 44.4, 39.9, 50.0), _box(0, 100, 100, 100, 100),
        _box(1, 210, 5, 215, 3)])
    for sr in (0, 1, 2, 3):
        c['sampling%d' % sr] = (2, 14, 14, 36, 7, 7, 1 / 16, sr, _random_rois([0, 1], 12, 224, 100 + sr).tolist())
    # large boxes at scale 1/8 (28 x 28 map of a 224 image): automatic grid of 3-4 samples per bin
    c['large_auto_grid'] = (2, 28, 28, 36, 7, 7, 1 / 8, 0, _random_rois([0, 1], 8, 224, 7, lo=0.0, span=0.1,
                                                                          min_w=150.0).tolist())
    c['ph7_pw14'] = (2, 14, 14, 36, 7, 14, 1 / 16, 0, _random_rois([0, 1], 6, 224, 8).tolist())
    c['ph3_pw5'] = (2, 14, 14, 36, 3, 5, 1 / 16, 2, _random_rois([0, 1], 6, 224, 9).tolist())
    c['pw32'] = (2, 14, 14, 36, 2, 32, 1 / 16, 0, _random_rois([0, 1], 5, 224, 10, span=0.9).tolist())
    c['h1'] = (2, 1, 9, 36, 7, 7, 1 / 16, 0, [_box(0, -10, -10, 140, 10), _box(1, 3, -20, 100, 30),
                                               _box(0, 20, 0, 60, 0)])
    c['w1'] = (2, 9, 1, 36, 7, 7, 1 / 16, 2, [_box(0, -10, -10, 10, 140), _box(1, -20, 3, 30, 100)])
    c['map2x2'] = (2, 2, 2, 36, 7, 7, 1 / 16, 0, [_box(0, -8, -8, 40, 40), _box(1, 4, 4, 20, 28),
                                                   _box(1, 0, 0, 31, 31)])
    c['c4'] = (2, 14, 14, 4, 7, 7, 1 / 16, 0, _random_rois([0, 1], 6, 224, 11).tolist())
    c['c2048'] = (2, 14, 14, 2048, 7, 7, 1 / 16, 0, _random_rois([0, 1], 6, 224, 12).tolist())
    c['r0'] = (2, 14, 14, 36, 7, 7, 1 / 16, 0, [])
    c['overlap64'] = (1, 14, 14, 36, 7, 7, 1 / 16, 0, _random_rois([0], 64, 224, 13, lo=40.0, span=0.3).tolist())
    # images 0 and 2 only: image 1 receives no gradient at all
    c['n3_images_0_2'] = (3, 14, 14, 36, 7, 7, 1 / 16, 0, _random_rois([0, 2], 9, 224, 14).tolist())
    # the head's production shape (R50 res5 map of two 224 x 224 clips)
    c['prod_r4'] = (2, 14, 14, 2048, 7, 7, 1 / 16, 0, _random_rois([0, 1], 4, 224, 15).tolist())
    c['prod_r16'] = (2, 14, 14, 2048, 7, 7, 1 / 16, 0, _random_rois([0, 1], 16, 224, 16).tolist())
    return c


ROI_CASES = _roi_cases()
TV_CASES = ['borders', 'outside', 'degenerate', 'sampling0', 'sampling1', 'sampling2', 'sampling3', 'large_auto_grid',
            'ph7_pw14', 'ph3_pw5', 'pw32', 'h1', 'w1', 'map2x2', 'overlap64', 'n3_images_0_2']


def roi_matrix(rois, N, H, W, PH, PW, scale, sr):
    """Dense fp64 A[(r, ph, pw), (n, y, x)] of legacy RoIAlign: the sample table's fp32 bilinear weights, in fp64,
    divided by the bin's sample count."""
    from oracle import roi_align_np
    R = len(rois)
    A = np.zeros((R * PH * PW, N * H * W))
    if R == 0:
        return A
    table = roi_align_np.sample_table(np.asarray(rois, np.float32), H, W, PH, PW, scale, sr)
    for r, t in enumerate(table):
        cnt = float(t['grid_h'] * t['grid_w'])
        pos = t['pos'].reshape(PH * PW, -1)
        w = t['w'].reshape(PH * PW, -1).astype(np.float64) / cnt
        rows = np.broadcast_to((r * PH * PW + np.arange(PH * PW))[:, None], pos.shape)
        ok = pos >= 0
        np.add.at(A, (rows[ok], t['batch'] * H * W + pos[ok]), w[ok])
    return A


@pytest.mark.parametrize('name', TV_CASES)
def test_roi_matrix_matches_torchvision_fp64(name):
    """CPU check of the reference: A @ feat equals torchvision.ops.roi_align(aligned=False) in float64, and so does
    A^T @ dout equal its autograd backward.  The box coordinates are dyadic, so fp32 (the table) and fp64
    (torchvision) sample coordinates differ only by the table's fp32 roundings of values below 32 (a few of
    2^-20 ~ 1e-6 each); they select the same pixels and move each bilinear weight by about that much (measured
    1.1e-6 on 'borders'), hence the bound 1e-5."""
    import torchvision
    N, Hh, Ww, C, PH, PW, scale, sr, rois = ROI_CASES[name]
    rois = [[r[0]] + [round(v * 4) / 4 for v in r[1:]] for r in rois]          # dyadic: exact in fp32 and fp64
    A = torch.from_numpy(roi_matrix(rois, N, Hh, Ww, PH, PW, scale, sr))
    g = torch.Generator().manual_seed(5)
    feat = torch.randn((N, 3, Hh, Ww), generator=g, dtype=torch.float64).requires_grad_(True)
    rt = torch.tensor(rois, dtype=torch.float64).reshape(-1, 5)
    out = torchvision.ops.roi_align(feat, rt, (PH, PW), scale, sr, False)
    ref = (A @ feat.detach().permute(0, 2, 3, 1).reshape(N * Hh * Ww, 3)).reshape(len(rois), PH, PW, 3)
    assert rel_err(ref.permute(0, 3, 1, 2), out) < 1e-5
    dout = torch.randn(out.shape, generator=g, dtype=torch.float64)
    out.backward(dout)
    dref = (A.t() @ dout.permute(0, 2, 3, 1).reshape(-1, 3)).reshape(N, Hh, Ww, 3)
    assert rel_err(dref.permute(0, 3, 1, 2), feat.grad) < 1e-5


@gpu
@pytest.mark.parametrize('name', list(ROI_CASES))
def test_roi_align_fwd_bwd_against_exact_linear_map(K, name):
    """Forward = A @ feat and backward = A^T @ dout (fp64) for every case.  The backward adds into a random dfeat:
    every element equals pattern + gradient, and elements that no RoI bin touches keep the pattern bit for bit."""
    N, Hh, Ww, C, PH, PW, scale, sr, rois = ROI_CASES[name]
    R = len(rois)
    A = roi_matrix(rois, N, Hh, Ww, PH, PW, scale, sr)
    At = torch.from_numpy(A)
    feat = torch.randn((N, Hh, Ww, C), generator=torch.Generator().manual_seed(21))
    dout = torch.randn((R, PH, PW, C), generator=torch.Generator().manual_seed(22))
    fwd_ref = (At @ feat.double().reshape(-1, C)).reshape(R, PH, PW, C)
    bwd_ref = (At.t() @ dout.double().reshape(-1, C)).reshape(N, Hh, Ww, C)
    rois_d = torch.tensor(rois, dtype=torch.float32).reshape(-1, 5).cuda()
    out = torch.full((R, PH, PW, C), float('nan'), device='cuda')
    K.roi_align_fwd(feat.cuda(), rois_d, out, scale, sr)
    pattern = torch.randn((N, Hh, Ww, C), generator=torch.Generator().manual_seed(23))
    pattern *= max(float(bwd_ref.abs().max()), 1.0)
    df = pattern.cuda()
    K.roi_align_bwd(dout.cuda(), rois_d, df, scale, sr)
    torch.cuda.synchronize()
    if R:
        assert rel_err(out, fwd_ref) < 1e-5
    empty_bins = torch.from_numpy(~A.any(1)).reshape(R, PH, PW)
    assert (out.cpu()[empty_bins] == 0).all(), 'a bin without samples must be exactly zero'
    df = df.cpu()
    assert rel_err(df.double() - pattern.double(), bwd_ref) < 1e-5
    untouched = torch.from_numpy(~A.any(0)).reshape(N, Hh, Ww)
    assert torch.equal(bits(df)[untouched], bits(pattern)[untouched])
    if name == 'n3_images_0_2':
        assert bool(untouched[1].all()) and torch.equal(bits(df[1]), bits(pattern[1]))
    if name == 'outside':
        assert bool(empty_bins[[0, 1, 3]].all()) and not bool(empty_bins[2].any())
    if name == 'borders':
        assert bool(empty_bins.any()) and not bool(empty_bins.all()), 'some bins lie entirely past the border'
    if R:
        assert float(bwd_ref.abs().max()) > 0


@gpu
def test_roi_align_bwd_rejects_pooled_width_33(K):
    """The backward keeps a RoI's x weights per thread for PW <= 32: PW = 33 is refused (VLFB_E_BADARG) before
    anything is launched."""
    from vlfb import libvlfb as L
    lib = L.load()
    dout = torch.randn((2, 2, 33, 8), device='cuda')
    rois = torch.tensor([[0, 0., 0., 100., 100.], [0, 10., 10., 200., 60.]], device='cuda')
    df = torch.randn((1, 14, 14, 8), device='cuda')
    before = df.clone()
    rc = lib.vlfb_roi_align_bwd(dout.data_ptr(), rois.data_ptr(), df.data_ptr(), 1, 14, 14, 8, 2, 2, 33, 1 / 16, 0,
                                K._stream())
    torch.cuda.synchronize()
    assert rc == -1 and b'bad argument' in lib.vlfb_last_error()
    assert torch.equal(df, before)


# -------------------------------------------------------------------------- accumulating GEMM
def _gemm(K, a, b, d, split=0, atomic=True, stream_k=0, engine=0, alpha=1.0, bias=None, tile_n=0, pair=-1):
    """vlfb_gemm_params_t for d[z] (+)= alpha * a[z] @ b[z]^T (+ bias): a [B, M, K], b [B, N, K], d [B, M, N], all
    dense, with the shared stream-K workspace."""
    from vlfb import libvlfb as L
    B, M, Kd = a.shape
    N = b.shape[1]
    p = L.GemmParams()
    p.M, p.N, p.K, p.batch, p.taps, p.split_k = M, N, Kd, B, 1, split
    p.a.ptr, p.a.kind, p.a.ld, p.a.batch_stride = a.data_ptr(), L.OP_DENSE_K, a.stride(1), a.stride(0) if B > 1 else 0
    p.b.ptr, p.b.kind, p.b.ld, p.b.batch_stride = b.data_ptr(), L.OP_DENSE_K, b.stride(1), b.stride(0) if B > 1 else 0
    p.d, p.ldd, p.d_batch_stride = d.data_ptr(), d.stride(1), d.stride(0) if B > 1 else 0
    p.alpha = alpha
    p.flags = L.EPI_ATOMIC if atomic else 0
    if bias is not None:
        p.col_bias = bias.data_ptr()
    w = K.gemm_workspace(d.device)
    p.workspace, p.workspace_bytes = w.data_ptr(), w.numel() * 4
    p.engine, p.tile_n, p.pair, p.stream_k = engine, tile_n, pair, stream_k
    return p


def _plan(p):
    from vlfb import libvlfb as L
    out = L.GemmPlan()
    assert L.load().vlfb_gemm_plan(ctypes.byref(p), 148, ctypes.byref(out)) == 0
    return out


def _run(K, p):
    from vlfb import libvlfb as L
    L.check(L.load().vlfb_gemm(ctypes.byref(p), K._stream()), 'vlfb_gemm')


def _counters_zero(K):
    return int(K.gemm_workspace(torch.device('cuda'))[:16384].view(torch.int32).abs().sum()) == 0


@gpu
@pytest.mark.parametrize('B,M,N,K_,tile_n', [(1, 128, 157, 12288, 128), (3, 136, 36, 16384, 32),
                                             (2, 130, 100, 8192, 64)])
def test_atomic_stream_k_fixup_ragged_n_bias_alpha_batch(K, B, M, N, K_, tile_n):
    """Atomic products with a ragged N (N % 16 != 0: the general epilogue), a bias, alpha != 1 and a batch, forced
    onto stream-K: the last unit to reach a shared tile sums all pieces in piece order and adds the tile to D once.
    D starts from a random pattern: D = pattern + alpha * A B^T + bias, the bias added exactly once, the same bits
    in every run, and the workspace arrival counters back at zero.  (Stream-K fix-ups need both operands staged by
    TMA, whose boxes are a 128-row A tile and a tile_n-row B tile: M >= 128 and N >= tile_n.  Smaller products run
    as whole tiles whatever the plan query says.)"""
    a, b = rnd((B, M, K_), 31).cuda(), rnd((B, N, K_), 32).cuda()
    bias = torch.randn(N).cuda()
    alpha = 0.75
    prod = torch.bmm(a.double(), b.double().transpose(1, 2))
    d0 = torch.randn((B, M, N), generator=torch.Generator().manual_seed(33)) * float(prod.abs().max())
    ref = d0.double() + alpha * prod.cpu() + bias.double().cpu()
    outs = []
    for _ in range(3):
        d = d0.cuda()
        p = _gemm(K, a, b, d, split=0, atomic=True, stream_k=1, alpha=alpha, bias=bias, tile_n=tile_n)
        pl = _plan(p)
        assert (pl.stream_k, pl.split_k) == (1, 1), 'the case must run as stream-K pieces'
        _run(K, p)
        torch.cuda.synchronize()
        outs.append(d.cpu())
        assert _counters_zero(K)
    assert rel_err(outs[0].double() - d0.double(), ref - d0.double()) < 2e-5
    for o in outs[1:]:
        assert torch.equal(bits(o), bits(outs[0]))


def _sweep_pairs(nkt):
    return [T for T in (147, 149, 295, 297) if T * nkt >= 2 * 148]


@gpu
@pytest.mark.parametrize('nkt', [2, 3, 4, 8, 15, 16, 17])
def test_stream_k_bounds_sweep(K, nkt):
    """Forced stream-K over tile counts T on either side of 148 and 2 x 148 SMs and K extents of nkt 32-deep chunks
    around the thresholds of make_bounds (pieces of at least 1 / 2 / 4 chunks at tile ends for nkt < 8 / < 16 /
    >= 16): one 128 x 32 tile per batch entry, so T = batch.  Both the plain epilogue (store, fix-up through the
    workspace) and the atomic one (split_k 0: fixed-order fix-up, then one addition into a random D)."""
    for T in _sweep_pairs(nkt):
        Kd = 32 * nkt
        a, b = rnd((T, 128, Kd), 40 + T).cuda(), rnd((T, 32, Kd), 41 + nkt).cuda()
        prod = torch.bmm(a.double(), b.double().transpose(1, 2)).cpu()
        d0 = torch.randn((T, 128, 32), generator=torch.Generator().manual_seed(T)) * float(prod.abs().max())
        for atomic in (False, True):
            d = d0.cuda() if atomic else torch.full((T, 128, 32), float('nan'), device='cuda')
            p = _gemm(K, a, b, d, split=0 if atomic else 1, atomic=atomic, stream_k=1, tile_n=32)
            pl = _plan(p)
            assert (pl.stream_k, pl.tiles, pl.units, pl.tile_n) == (1, T, 148, 32), (T, nkt, atomic)
            _run(K, p)
            torch.cuda.synchronize()
            got = d.cpu().double() - (d0.double() if atomic else 0)
            assert rel_err(got, prod) < 2e-5, (T, nkt, atomic)
            assert _counters_zero(K), (T, nkt, atomic)


@gpu
def test_conv1_weight_gradient_at_production_size(K):
    """conv1's weight gradient at 2 x 32 x 224 x 224 (K = 802816 positions per temporal tap, the largest reduction of
    the step, spread as stream-K pieces over all SMs), on the W-padded clip the workspace feeds, with the padding-lane
    mask, added into a non-zero dw: equal to the fp64 cuDNN gradient, padding lanes untouched, and bit-identical on a
    second run.

    Bound: the error of a tensor-core product grows linearly with the length L of the accumulation one unit does
    (measured rel err ~2.4e-9 * L: whole 128-row tiles of L = 12288 and 16384 gave 2.9e-5 and 4.0e-5), as for an
    accumulator that truncates at each K = 8 step: error <= sum over L/8 steps of 2^-23 |partial sum|, which for
    random operands is ~2^-23 * L / 48 of the largest result.  Here a unit's piece is L = 32 * ceil(5 * 25088 / 148)
    = 27136 (measured 6.7e-5); the bound is 2^-23 * L / 16, three times the estimate."""
    from vlfb import libvlfb as L
    K.set_gemm_backend('tcgen05')
    N, T, S = 2, 32, 224
    g = K.conv_geom((N, T, S, S, 4), 64, (5, 7, 7), (1, 2, 2), (2, 3, 3))
    x = rnd((N, 3, T, S, S), 61)
    left, pitch = 3, (3 + S + 5 + 3) // 4 * 4
    buf = torch.zeros((N, T, S, pitch, 4), device='cuda')
    K.nc_to_cl(x.cuda().contiguous(), buf, N, 3, T * S * S, 4, tf32_out=True, width=S, pitch=pitch, left=left)
    x4 = buf[:, :, :, left:left + S, :]
    dy = rnd(K.out_shape(g), 62).cuda()
    p = L.GemmParams()
    p.M, p.N, p.K, p.batch, p.taps, p.split_k, p.flags = 64, 7 * 32, N * T * g.Ho * g.Wo, 1, 5, 0, L.EPI_ATOMIC
    p.a.kind, p.b.kind = L.OP_DENSE_MN, L.OP_STEM_MN
    w = K.gemm_workspace(dy.device)
    p.workspace, p.workspace_bytes = w.data_ptr(), w.numel() * 4
    pl = _plan(p)
    assert (pl.stream_k, pl.split_k) == (1, 1)
    # fp64 reference on the GPU (cuDNN double), independent of libvlfb
    xd = x.cuda().double()
    dyd = dy.double().permute(0, 4, 1, 2, 3)
    ref = torch.nn.grad.conv3d_weight(xd, (64, 3, 5, 7, 7), dyd, (1, 2, 2), (2, 3, 3)).cpu()
    del xd, dyd
    ref = stem_pack(ref)
    mask = torch.ones((8, 4))
    mask[7, :] = 0
    mask[:, 3] = 0
    pad = (mask == 0).expand(64, 5, 7, 8, 4)
    dw0 = torch.randn((64, 5, 7, 8, 4), generator=torch.Generator().manual_seed(63)) * float(ref.abs().max())
    outs = []
    for _ in range(2):
        dw = dw0.cuda()
        K.conv_wgrad(dy, x4, dw, g, col_mask=mask.reshape(32).cuda())
        torch.cuda.synchronize()
        outs.append(dw.cpu())
    err = rel_err(outs[0].double() - dw0.double(), ref)
    print('conv1 wgrad at 2x32x224x224: rel err %.2e' % err)
    piece = 32 * -(-5 * (p.K // 32) // 148)
    assert err < 2.0 ** -23 * piece / 16
    assert torch.equal(bits(outs[0])[pad], bits(dw0)[pad])
    assert torch.equal(bits(outs[0]), bits(outs[1]))
    assert _counters_zero(K)


@gpu
@pytest.mark.parametrize('case', ['tcgen05_whole_tiles', 'simt_k4100', 'simt_fallback_unaligned'])
def test_library_split_equals_explicit_single_slice(K, case):
    """vlfb.h: an atomic product with split_k == 0, a workspace and stream_k >= 0 is never split into K slices that
    add into d in arrival order.  When its plan is one K slice without stream-K, it must therefore give exactly the
    bits of an explicit split_k = 1 call -- on the tensor-core engine, on the SIMT engine, and when the library sends
    a product to SIMT because an operand is not 16-byte addressable."""
    from vlfb import libvlfb as L
    # T tiles x nkt chunks < 2 x 148 for every tile width: never worth stream-K, so the plan is whole tiles
    B, M, N, Kd, engine, offset = {'tcgen05_whole_tiles': (1, 128, 64, 2048, L.ENGINE_TCGEN05, 0),
                                   'simt_k4100': (1, 8, 64, 4100, L.ENGINE_SIMT, 0),
                                   'simt_fallback_unaligned': (1, 4, 64, 4096, L.ENGINE_TCGEN05, 1)}[case]
    # `offset` floats in front of the operand: its address is 4 bytes past a 16-byte boundary
    a_buf = rnd((B * M * Kd + offset,), 71).cuda()
    a = a_buf[offset:].view(B, M, Kd)
    b = rnd((B, N, Kd), 72).cuda()
    bias = torch.randn(N).cuda()
    ref = torch.bmm(a.double(), b.double().transpose(1, 2)).cpu() + bias.double().cpu()
    d0 = torch.randn((B, M, N), generator=torch.Generator().manual_seed(73)) * float(ref.abs().max())
    got = {}
    for split in (0, 1):
        d = d0.cuda()
        p = _gemm(K, a, b, d, split=split, atomic=True, engine=engine, bias=bias, pair=0)
        if split == 0:
            pl = _plan(p)
            assert (pl.split_k, pl.stream_k) == (1, 0), case
        _run(K, p)
        torch.cuda.synchronize()
        got[split] = d.cpu()
    assert rel_err(got[0].double() - d0.double(), ref) < 2e-5
    assert torch.equal(bits(got[0]), bits(got[1])), 'split_k = 0 cut the product into atomic K slices'


# -------------------------------------------------------------------------- colsum
@gpu
def test_colsum_short_workspace_is_refused(K):
    """A workspace 4 bytes short of vlfb_colsum_workspace_bytes() returns VLFB_E_WORKSPACE with a message naming
    the workspace, and leaves out unchanged."""
    from vlfb import libvlfb as L
    lib = L.load()
    rows, cols = 5000, 80
    need = int(lib.vlfb_colsum_workspace_bytes(rows, cols))
    assert need > 0
    x = torch.randn((rows, cols), device='cuda')
    out = torch.randn(cols, device='cuda')
    before = out.clone()
    ws = torch.zeros(need // 4, device='cuda')
    rc = lib.vlfb_colsum(x.data_ptr(), cols, out.data_ptr(), rows, cols, 1, ws.data_ptr(), need - 4, K._stream())
    torch.cuda.synchronize()
    assert rc == -4 and b'workspace' in lib.vlfb_last_error()
    assert torch.equal(out, before)


# -------------------------------------------------------------------------- a whole training step
TINY = ['NUM_GPUS', 1, 'TRAIN.BATCH_SIZE', 2, 'TRAIN.CROP_SIZE', 64, 'TRAIN.VIDEO_LENGTH', 8,
        'TEST.BATCH_SIZE', 2, 'TEST.CROP_SIZE', 64, 'TEST.VIDEO_LENGTH', 8, 'LFB.WINDOW_SIZE', 4,
        'TRAIN.DROPOUT_RATE', 0.0, 'FBO_NL.INPUT_DROPOUT_ON', False, 'FBO_NL.LFB_DROPOUT_ON', False]
FULL = ['NUM_GPUS', 1, 'TRAIN.BATCH_SIZE', 2, 'TEST.BATCH_SIZE', 2,
        'TRAIN.DROPOUT_RATE', 0.0, 'FBO_NL.INPUT_DROPOUT_ON', False, 'FBO_NL.LFB_DROPOUT_ON', False]


@pytest.fixture
def ws():
    from vlfb import kernels, workspace
    assert torch.cuda.is_available()
    kernels.set_gemm_backend('tcgen05')
    workspace.ResetWorkspace()
    yield workspace
    workspace.ResetWorkspace()


@gpu
@pytest.mark.parametrize('size', ['tiny', 'full_config2'])
def test_training_step_is_bit_identical_run_after_run(ws, size):
    """The AVA R50-I3D-NL + FBO-NL train step (update ops removed), run eagerly twice and then replayed twice from
    its captured CUDA graph: loss, pred and every trainable gradient have the same bits in all four runs.  The first
    eager run does not yet know how many contributions each gradient has, so it cannot fold the last one into a dgrad
    epilogue; with the deferred two-term sums (executor.LAZY_GRAD_SUM) a three-term sum would then be associated
    differently from the later runs, so they are off here, as in test_gpu_model.py's grad-finish test."""
    from oracle import model as OM
    from vlfb import executor as X
    ov, crop, frames = (TINY, 64, 8) if size == 'tiny' else (FULL, 224, 32)
    H.setup_cfg('ava_r50_lfb_nl.yaml', ov)
    ocfg = H.oracle_cfg('ava_r50_lfb_nl.yaml', ov)
    params = OM.make_params(ocfg, seed=2)
    inputs = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=2, crop=crop, frames=frames)
    model, sfx = H.build('train', True)
    H.feed_params(params)
    H.feed_inputs(inputs, sfx)
    name = model.net.Proto().name
    net = ws.current().nets[name]
    net.update_ops = []
    lazy0, X.LAZY_GRAD_SUM = X.LAZY_GRAD_SUM, False
    runs = []
    try:
        for _ in range(4):
            ws.RunNet(name)
            torch.cuda.synchronize()
            blobs = dict((n + '_grad', ws.FetchBlob('gpu_0/' + n + '_grad').copy()) for n in model.TrainableParams())
            blobs['loss'] = np.asarray(ws.FetchBlob('gpu_0/loss'), np.float32).copy()
            blobs['pred'] = ws.FetchBlob('gpu_0/pred').copy()
            runs.append(blobs)
    finally:
        X.LAZY_GRAD_SUM = lazy0
    assert len(net._graphs) == 1, 'runs 3 and 4 should have been graph replays'
    assert len(runs[0]) > 100 and np.abs(runs[0]['conv1_w_grad']).max() > 0
    for rep in (1, 2, 3):
        differ = [n for n in runs[0] if not np.array_equal(runs[rep][n].view(np.int32), runs[0][n].view(np.int32))]
        assert not differ, (rep, differ[:10])
