"""CPU tests of the oracle itself (what pins it, given that the reference has no tests and cannot
run here -- DESIGN.md section 2) and of the host-side config / LR logic."""
import os

import numpy as np
import pytest
import torch

import harness as H

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
TINY = ['NUM_GPUS', 1, 'TRAIN.BATCH_SIZE', 2, 'TRAIN.CROP_SIZE', 64, 'TRAIN.VIDEO_LENGTH', 8,
        'LFB.WINDOW_SIZE', 4, 'TRAIN.DROPOUT_RATE', 0.0, 'FBO_NL.INPUT_DROPOUT_ON', False,
        'FBO_NL.LFB_DROPOUT_ON', False]


def test_numpy_roi_align_matches_torchvision_legacy_mode():
    import torchvision
    from oracle import roi_align_np
    g = torch.Generator().manual_seed(0)
    feat = torch.randn((2, 8, 14, 14), generator=g)
    rois = torch.tensor([[0, 0., 0., 223., 223.], [1, 10.5, 20.25, 100.75, 180.5], [0, 3.3, 4.4, 3.9, 5.0],
                         [1, 111., 7., 223., 60.]])
    ref = torchvision.ops.roi_align(feat, rois, (7, 7), 1.0 / 16, 0, False).numpy()
    mine = roi_align_np.roi_align(feat.numpy(), rois.numpy())
    assert np.abs(ref - mine).max() < 1e-6


def test_roi_table_golden_is_stable():
    from oracle import roi_align_np
    z = np.load(os.path.join(GOLD, 'roi_table_14x14.npz'))
    table = roi_align_np.sample_table(z['rois'], 14, 14, 7, 7, 1.0 / 16, 0)
    for i, t in enumerate(table):
        assert tuple(z['grid'][i]) == (t['grid_h'], t['grid_w'])
        assert np.array_equal(z['pos%d' % i], t['pos'])
        assert np.array_equal(z['w%d' % i].view(np.int32), t['w'].view(np.int32))
    # hand-checkable facts: the full-frame box on a 14x14 map -> bins of 13.9375/7, 2x2 samples per bin
    assert tuple(z['grid'][0]) == (2, 2) and tuple(z['grid'][2]) == (1, 1)


def test_parameter_inventory_matches_survey():
    """SURVEY.md section 8a: 123 trainable tensors / 39.96 M params (R50 + FBO-3L), 63.6 M (R101)."""
    from oracle import model as OM
    for yaml_name, n_tensors, n_params in (('ava_r50_lfb_nl_3l.yaml', 123, 39.98e6),
                                           ('ava_r101_lfb_nl_3l.yaml', 174, 63.6e6)):
        spec = OM.param_spec(H.oracle_cfg(yaml_name, []))
        tr = [(k, s) for k, (s, kind) in spec.items() if kind not in ('affine_s', 'affine_b')]
        assert len(tr) == n_tensors
        assert abs(sum(int(np.prod(s)) for _, s in tr) - n_params) / n_params < 0.01


def test_known_answer_ops():
    from oracle import ops as O
    # AffineNd (affine_nd_op.cu:32-58)
    x = torch.arange(2 * 3 * 2, dtype=torch.float32).view(2, 3, 2, 1, 1)
    s, b = torch.tensor([1., 2., 3.]), torch.tensor([0., 1., -1.])
    y = O.affine_nd(x, s, b)
    assert y[1, 2, 1, 0, 0].item() == 11 * 3 - 1 and O.affine_nd_grad(x, s)[0, 1, 0, 0, 0].item() == 4.0
    # BN fold + inflation (checkpoints.py:108-110,359-362)
    sc, bi = O.bn_fold(np.array([2.]), np.array([1.]), np.array([3.]), np.array([4. - 1e-5]))
    assert abs(sc[0] - 1.0) < 1e-9 and abs(bi[0] + 2.0) < 1e-9
    w3 = O.inflate_2d_to_3d(np.ones((4, 3, 7, 7)), 5)
    assert w3.shape == (4, 3, 5, 7, 7) and abs(w3.sum() - 4 * 3 * 49) < 1e-9
    # Nesterov (model_builder_video.py:375-388): m' = mu*m + lr*(g+wd*p); p -= (1+mu)*m' - mu*m
    p, m = O.nesterov_update(torch.tensor([1.0]), torch.tensor([0.5]), torch.tensor([0.2]), 0.1, 0.9, 0.01)
    assert abs(m.item() - (0.18 + 0.1 * 0.51)) < 1e-7 and abs(p.item() - (1 - (1.9 * 0.231 - 0.18))) < 1e-7
    # Detectron sigmoid CE: ignores -1, normalises by #valid
    l = O.sigmoid_cross_entropy_loss(torch.tensor([[0.0, 100.0]]), torch.tensor([[1, -1]]), 2.0)
    assert abs(l.item() - 2 * np.log(2.0)) < 1e-6
    # LayerNorm axis=1 without affine
    yln, mean, std = O.layer_norm_axis1(torch.tensor([[1., 3.], [2., 2.]]).view(2, 2, 1, 1, 1))
    assert torch.allclose(yln[0].view(-1), torch.tensor([-1., 1.]), atol=1e-4) and float(yln[1].abs().max()) == 0.0


def test_oracle_regression_golden():
    from oracle import model as OM
    z = np.load(os.path.join(GOLD, 'tiny_ava_fbo_nl.npz'))
    ocfg = H.oracle_cfg('ava_r50_lfb_nl.yaml', TINY)
    params = OM.make_params(ocfg, seed=2)
    inputs = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=2, crop=64, frames=8)
    blobs, prob, loss = OM.forward(ocfg, params, inputs, 'train')
    assert abs(loss.item() - float(z['loss'])) < 1e-4 * abs(float(z['loss']))
    for b in ('box_pooled', 'pool5', 'pred'):
        assert H.rel(blobs[b].detach().numpy(), z['blob/' + b]) < 1e-4


def test_lr_policy_and_config_merge():
    from core.config import config as cfg
    from utils import lr_policy
    H.setup_cfg('ava_r50_lfb_nl_3l.yaml', [])
    assert cfg.LFB.NUM_LFB_FEAT == 300 and cfg.SOLVER.STEPS == [0, 100000, 120000, 140000]
    assert cfg.FBO_NL.NUM_LAYERS == 3
    assert abs(lr_policy.get_lr_at_iter(0) - 0.01) < 1e-7                 # warm-up start
    assert abs(lr_policy.get_lr_at_iter(1999) - 0.04) < 1e-6              # warm-up end
    assert abs(lr_policy.get_lr_at_iter(50000) - 0.04) < 1e-7
    assert abs(lr_policy.get_lr_at_iter(110000) - 0.004) < 1e-7
    from core import config as C
    with pytest.raises(KeyError):
        C.merge_dicts({'NOT_A_KEY': 1}, cfg)
    with pytest.raises(ValueError):
        C.merge_dicts({'NUM_GPUS': 'eight'}, cfg)


def test_reference_yaml_files_load():
    """Every config the reference ships (copied unchanged into tests/golden/reference_configs) loads and validates."""
    import glob
    from core import config as C
    files = sorted(glob.glob(os.path.join(GOLD, 'reference_configs', '*.yaml')))
    for f in files:
        C.reset_cfg()
        C.cfg_from_file(f)
        C.assert_and_infer_cfg()
    assert len(files) >= 26


def test_oracle_ops_agree_with_independent_implementations():
    """The reference ships no golden vectors and Caffe2 cannot run here ("parity unpinned", DESIGN section 2); what CAN be
    pinned is every restated operator that has an independent implementation of the same published definition in
    PyTorch: LayerNorm, sigmoid / softmax cross-entropy, Nesterov SGD with weight decay (Caffe2's lr-folded momentum form
    against torch.optim.SGD over several steps), pooling, softmax, batched matmul.  (RoIAlign: torchvision, above;
    SpatialBN: F.batch_norm, tests/test_spatial_bn.py.)"""
    import torch.nn.functional as F
    from oracle import ops as O
    g = torch.Generator().manual_seed(7)
    x = torch.randn((5, 512, 1, 1, 1), generator=g, dtype=torch.float64) * 3 + 1
    y, mean, std = O.layer_norm_axis1(x, eps=1e-5)
    assert (y.reshape(5, 512) - F.layer_norm(x.reshape(5, 512), (512,), eps=1e-5)).abs().max() < 1e-12
    assert (std.view(-1) - torch.sqrt(x.reshape(5, -1).var(dim=1, unbiased=False) + 1e-5)).abs().max() < 1e-12
    # Detectron SigmoidCrossEntropyLoss: sum over the valid elements / #valid * scale; targets -1 are ignored
    logits = torch.randn((6, 80), generator=g, dtype=torch.float64) * 4
    t = (torch.rand((6, 80), generator=g) < 0.1).to(torch.int32)
    t[1, :7] = -1
    valid = t != -1
    ref = F.binary_cross_entropy_with_logits(logits[valid], t[valid].double(), reduction='sum') / valid.sum() * 0.125
    assert abs(float(O.sigmoid_cross_entropy_loss(logits, t, scale=0.125) - ref)) < 1e-12
    labels = torch.randint(0, 80, (6,), generator=g)
    prob, loss = O.softmax_with_loss(logits, labels, scale=0.5)
    assert abs(float(loss - 0.5 * F.cross_entropy(logits, labels))) < 1e-12
    assert (prob - torch.softmax(logits, dim=1)).abs().max() < 1e-15
    # WeightedSum + MomentumSGDUpdate(nesterov) == torch.optim.SGD(nesterov, weight_decay) at constant lr, 4 steps
    p0 = torch.randn(257, generator=g, dtype=torch.float64)
    grads = [torch.randn(257, generator=g, dtype=torch.float64) for _ in range(4)]
    p, m = p0.clone(), torch.zeros_like(p0)
    tp = p0.clone().requires_grad_(True)
    opt = torch.optim.SGD([tp], lr=0.03, momentum=0.9, nesterov=True, weight_decay=1e-4)
    for gr in grads:
        p, m = O.nesterov_update(p, gr, m, 0.03, 0.9, 1e-4)
        tp.grad = gr.clone()
        opt.step()
    assert (p - tp.detach()).abs().max() < 1e-13
    # pooling / softmax(axis=2) / BatchMatMul(trans_a, trans_b)
    v = torch.randn((2, 8, 4, 9, 9), generator=g, dtype=torch.float64)
    assert torch.equal(O.max_pool_nd(v, (1, 3, 3), (1, 2, 2), (0, 1, 1)), F.max_pool3d(v, (1, 3, 3), (1, 2, 2), (0, 1, 1)))
    assert (O.avg_pool_nd(v, (4, 1, 1), (1, 1, 1), (0, 0, 0)) - v.mean(dim=2, keepdim=True)).abs().max() < 1e-14
    a3 = torch.randn((3, 5, 7), generator=g, dtype=torch.float64)
    assert (O.softmax_axis2(a3) - torch.softmax(a3, dim=2)).abs().max() < 1e-15
    b3 = torch.randn((3, 5, 4), generator=g, dtype=torch.float64)
    assert (O.batch_matmul(a3, b3, trans_a=1) - torch.einsum('bkm,bkn->bmn', a3, b3)).abs().max() < 1e-13
    c3 = torch.randn((3, 4, 7), generator=g, dtype=torch.float64)
    assert (O.batch_matmul(a3, c3, trans_b=1) - torch.einsum('bmk,bnk->bmn', a3, c3)).abs().max() < 1e-13
