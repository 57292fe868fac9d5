"""GPU parity of the whole hot path through the builder API + workspace (C ABI underneath):
R50-I3D-NL (+FBO) forward / backward / SGD step on cuda:0 versus the fp64 oracle.

Tolerances.  The contractions run on tcgen05 kind::tf32 (10-bit mantissa operands, fp32
accumulate).
  * Forward outputs vs the PLAIN fp64 oracle: the north-star bound 1e-3 (max|a-b|/max|b|).
  * Gradients: a TF32-level perturbation (5e-4 relative) of an activation flips ReLUs / LayerNorm->ReLU
    outputs that lie within that distance of zero and moves max-pool / RoI-max arg-maxes between
    near-equal candidates, which re-routes the gradient of the affected channel completely.  This is
    a property of the function at TF32 operand precision, not of the kernels: the fp32 SIMT engine
    shows the same level (measured 1.7e-1 max-norm on res5_1_branch2c_w), and even an oracle that
    emulates the TF32 roundings cannot be made bit-identical (profiles/r01_grad_parity_notes.md).
    Gradients are therefore held to a relative L2 error <= 0.15 and cosine >= 0.98 per tensor and a
    median relative L2 over all tensors <= 2e-2.  What pins the backward pass exactly:
    tests/test_engine_cpu.py (same host logic in fp64 vs the oracle, 1e-7 on every parameter) and
    tests/test_gpu_kernels.py (every dgrad / wgrad kernel vs fp64, 2e-5).
"""
import os

import numpy as np
import pytest
import torch

import harness as H

pytestmark = pytest.mark.gpu

TINY = ['NUM_GPUS', 1, 'TRAIN.BATCH_SIZE', 2, 'TRAIN.CROP_SIZE', 64, 'TRAIN.VIDEO_LENGTH', 8,
        'TEST.BATCH_SIZE', 2, 'TEST.CROP_SIZE', 64, 'TEST.VIDEO_LENGTH', 8, 'LFB.WINDOW_SIZE', 4,
        'TRAIN.DROPOUT_RATE', 0.0, 'FBO_NL.INPUT_DROPOUT_ON', False, 'FBO_NL.LFB_DROPOUT_ON', False]
FULL = ['NUM_GPUS', 1, 'TRAIN.BATCH_SIZE', 2, 'TEST.BATCH_SIZE', 2,
        'TRAIN.DROPOUT_RATE', 0.0, 'FBO_NL.INPUT_DROPOUT_ON', False, 'FBO_NL.LFB_DROPOUT_ON', False]
FWD_BLOBS = ['box_pooled', 'pool5', 'pred', 'prob']
FWD_TOL = 1e-3
GRAD_L2_TOL = 0.15
GRAD_COS_TOL = 0.98
GRAD_MEDIAN_L2_TOL = 2e-2


@pytest.fixture
def ws():
    from vlfb import kernels, workspace
    assert torch.cuda.is_available()
    kernels.set_gemm_backend('tcgen05')
    workspace.ResetWorkspace()
    yield workspace
    workspace.ResetWorkspace()


def _oracle(ocfg, params, inputs, split, backward, emulate_tf32=False):
    from oracle import model as OM
    p64 = dict((k, v.double().requires_grad_(backward)) for k, v in params.items())
    i64 = dict((k, (v.double() if v.dtype == torch.float32 else v)) for k, v in inputs.items())
    blobs, prob, loss = OM.forward(ocfg, p64, i64, split, emulate_tf32=emulate_tf32)
    if backward:
        loss.backward()
    return p64, blobs, loss


def _train_case(ws, yaml_name, overrides, crop, frames, rois_per_clip, backend='tcgen05', check_all_grads=True,
                median_tol=GRAD_MEDIAN_L2_TOL):
    from oracle import model as OM
    from vlfb import kernels
    kernels.set_gemm_backend(backend)
    H.setup_cfg(yaml_name, overrides)
    ocfg = H.oracle_cfg(yaml_name, overrides)
    params = OM.make_params(ocfg, seed=2)
    inputs = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=rois_per_clip, crop=crop, frames=frames)
    model, sfx = H.build('train', True)
    H.feed_params(params)
    H.feed_inputs(inputs, sfx)
    p64, blobs, loss = _oracle(ocfg, params, inputs, 'train', True)
    net = ws.current().nets[model.net.Proto().name]
    upd, net.update_ops = net.update_ops, []
    ws.RunNet(model.net.Proto().name)
    torch.cuda.synchronize()
    net.update_ops = upd
    report = {}
    report['loss'] = H.rel(ws.FetchBlob('gpu_0/loss'), loss.item())
    for b in FWD_BLOBS:
        if b in blobs:
            report[b] = H.rel(ws.FetchBlob('gpu_0/' + b), blobs[b].detach().numpy())
    gerr, gcos = {}, {}
    names = model.TrainableParams() if check_all_grads else [
        'pred_w', 'lfb_1x1_w', 'lfb_nl1_out_w', 'res5_2_branch2c_w', 'res4_3_branch2b_w', 'nonlocal_conv4_1_theta_w',
        'nonlocal_conv3_1_out_w', 'res2_0_branch2a_w', 'conv1_w']
    for name in names:
        if name not in p64:
            continue
        ref = p64[name].grad.numpy()
        g = ws.FetchBlob('gpu_0/' + name + '_grad')
        nref = float(np.linalg.norm(ref.astype(np.float64)))
        if nref < 1e-7:
            continue                                    # e.g. phi_b: mathematically zero gradient
        g64 = g.astype(np.float64)
        gerr[name] = float(np.linalg.norm(g64 - ref) / nref)
        gcos[name] = float((g64 * ref).sum() / (np.linalg.norm(g64) * nref + 1e-30))
    worst = sorted(gerr.items(), key=lambda kv: -kv[1])[:5]
    med = float(np.median(list(gerr.values())))
    print('\n[%s %s crop %d] forward rel err vs oracle: %s\n   grads: median rel-L2 %.2e, worst %s, min cos %.4f' % (
        yaml_name, backend, crop, ' '.join('%s=%.2e' % kv for kv in report.items()), med,
        ' '.join('%s=%.2e' % kv for kv in worst), min(gcos.values())))
    for k, v in report.items():
        assert v < FWD_TOL, (k, v)
    for k, v in gerr.items():
        assert v < GRAD_L2_TOL and gcos[k] > GRAD_COS_TOL, (k, v, gcos[k])
    assert med < median_tol, med
    return model, params, p64


def test_tiny_fbo_nl_train_step(ws):
    _train_case(ws, 'ava_r50_lfb_nl.yaml', TINY, 64, 8, 2)


def test_tiny_gradients_vs_tf32_emulating_oracle(ws):
    """Second, independent gradient oracle: `emulate_tf32` rounds operands at the same graph points as the engine
    (tests/test_engine_cpu.py proves the two coincide exactly in fp64).  In fp32 on the GPU the accumulation
    order perturbs values by ~1e-7, which moves ~0.3% of the elements of every layer across a TF32 rounding
    boundary (measured: pool1 2.8e-3 of the elements, 39% after 8 blocks), so the two still differ by TF32
    noise; the test therefore bounds the same norms as the plain-oracle test, it does not demand bit patterns."""
    from oracle import model as OM
    H.setup_cfg('ava_r50_lfb_nl.yaml', TINY)
    ocfg = H.oracle_cfg('ava_r50_lfb_nl.yaml', TINY)
    params = OM.make_params(ocfg, seed=2)
    inputs = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=2, crop=64, frames=8)
    model, sfx = H.build('train', True)
    H.feed_params(params)
    H.feed_inputs(inputs, sfx)
    p64, blobs, loss = _oracle(ocfg, params, inputs, 'train', True, emulate_tf32=True)
    net = ws.current().nets[model.net.Proto().name]
    net.update_ops = []
    ws.RunNet(model.net.Proto().name)
    for b in ['pool1', 'res3_3_branch2c_bn', 'res5_2_branch2c_bn', 'box_pooled', 'pool5', 'pred']:
        a, r = ws.FetchBlob('gpu_0/' + b), blobs[b].detach().numpy()
        frac = float((np.abs(a - r) > 2e-5 * np.abs(r).max()).mean())
        print('%s: %.2e of the elements differ from the emulating oracle (max-norm %.2e)' % (b, frac, H.rel(a, r)))
        assert H.rel(a, r) < 3e-3, (b, H.rel(a, r))
    errs, coss = {}, {}
    for name in model.TrainableParams():
        ref = p64[name].grad.numpy()
        nref = float(np.linalg.norm(ref))
        if nref < 1e-7:
            continue
        g = ws.FetchBlob('gpu_0/' + name + '_grad').astype(np.float64)
        errs[name] = float(np.linalg.norm(g - ref) / nref)
        coss[name] = float((g * ref).sum() / (np.linalg.norm(g) * nref))
    worst = sorted(errs.items(), key=lambda kv: -kv[1])[:6]
    print('grads vs emulating oracle: median rel-L2 %.2e, worst %s, min cos %.5f' % (
        float(np.median(list(errs.values()))), ' '.join('%s=%.2e' % kv for kv in worst), min(coss.values())))
    assert float(np.median(list(errs.values()))) < GRAD_MEDIAN_L2_TOL
    for k, v in errs.items():
        assert v < GRAD_L2_TOL and coss[k] > GRAD_COS_TOL, (k, v, coss[k])


def test_grad_finish_fusion_and_graph_replay_agree_with_first_run(ws):
    """Run 1 = separate ReLU-backward / rounding passes; run 2 = folded into the last dgrad GEMM's epilogue
    (executor "grad finish" fusion); run 3+ = the captured CUDA graph.  Same arithmetic, and every reduction sums in
    a fixed order, so the gradients are bit-identical."""
    from oracle import model as OM
    from vlfb import executor as X
    H.setup_cfg('ava_r50_lfb_nl.yaml', TINY)
    ocfg = H.oracle_cfg('ava_r50_lfb_nl.yaml', TINY)
    params = OM.make_params(ocfg, seed=2)
    inputs = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=2, crop=64, frames=8)
    model, sfx = H.build('train', True)
    H.feed_params(params)
    H.feed_inputs(inputs, sfx)
    net = ws.current().nets[model.net.Proto().name]
    net.update_ops = []
    runs = []
    fuse0, X.FUSE_GRAD_FINISH = X.FUSE_GRAD_FINISH, True       # (the default since round 2)
    lazy0, X.LAZY_GRAD_SUM = X.LAZY_GRAD_SUM, False            # same association of three-term sums in every run
    for rep in range(4):
        n0 = X.STATS['fused_grad_finish']
        ws.RunNet(model.net.Proto().name)
        torch.cuda.synchronize()
        if rep < 2:
            assert (X.STATS['fused_grad_finish'] - n0 > 40) == (rep == 1)
        runs.append(dict((n, ws.FetchBlob('gpu_0/' + n + '_grad').copy()) for n in model.TrainableParams()))
    X.FUSE_GRAD_FINISH, X.LAZY_GRAD_SUM = fuse0, lazy0
    assert len(net._graphs) == 1, 'the step should have been captured into a CUDA graph by now'
    for rep in (1, 2, 3):
        differ = [n for n in runs[0] if not np.array_equal(runs[rep][n].view(np.int32), runs[0][n].view(np.int32))]
        assert not differ, (rep, differ[:10])


def test_enqueue_blobs_matches_feed_blob(ws):
    """Asynchronous feeding (copy stream + staging slots + dequeue at RunNet) gives the same step as FeedBlob,
    batch after batch, including after the step has been captured into a CUDA graph."""
    from oracle import model as OM
    H.setup_cfg('ava_r50_lfb_nl.yaml', TINY)
    ocfg = H.oracle_cfg('ava_r50_lfb_nl.yaml', TINY)
    params = OM.make_params(ocfg, seed=2)
    model, sfx = H.build('train', True)
    H.feed_params(params)
    net = ws.current().nets[model.net.Proto().name]
    net.update_ops = []
    batches = [OM.make_inputs(ocfg, n_clips=2, rois_per_clip=2, crop=64, frames=8, seed=50 + i) for i in range(4)]
    want = []
    for b in batches:
        H.feed_inputs(b, sfx)
        ws.RunNet(model.net.Proto().name)
        want.append((float(ws.FetchBlob('gpu_0/loss')), ws.FetchBlob('gpu_0/pred').copy()))
    assert len(set(w[0] for w in want)) == 4, 'the batches must differ'
    host = [dict(('gpu_0/%s%s' % (k, sfx), v.contiguous().pin_memory()) for k, v in b.items()) for b in batches]
    ws.EnqueueBlobs(host[0])
    for i in range(4):
        ws.RunNet(model.net.Proto().name)
        if i + 1 < 4:
            ws.EnqueueBlobs(host[i + 1])             # overlaps the step that is running
        assert abs(float(ws.FetchBlob('gpu_0/loss')) - want[i][0]) <= 1e-6 * abs(want[i][0])
        assert H.rel(ws.FetchBlob('gpu_0/pred'), want[i][1]) < 1e-6
    # pipelined read-back: step i's loss / pred are collected after step i+1 has been launched
    ws.EnqueueBlobs(host[0])
    pending = None
    got = []
    for i in range(4):
        ws.RunNet(model.net.Proto().name)
        if i + 1 < 4:
            ws.EnqueueBlobs(host[i + 1])
        nxt = (ws.FetchBlobAsync('gpu_0/loss'), ws.FetchBlobAsync('gpu_0/pred'))
        if pending is not None:
            got.append((float(pending[0].get()), pending[1].get()))
        pending = nxt
    got.append((float(pending[0].get()), pending[1].get()))
    for i in range(4):
        assert abs(got[i][0] - want[i][0]) <= 1e-6 * abs(want[i][0])
        assert got[i][1].shape == want[i][1].shape and H.rel(got[i][1], want[i][1]) < 1e-6


def test_tiny_simt_engine_agrees(ws):
    """Same graph on the SIMT fp32 engine: isolates TF32 effects from logic errors."""
    _train_case(ws, 'ava_r50_lfb_nl.yaml', TINY, 64, 8, 2, backend='simt')


def test_tiny_charades_variant(ws):
    _train_case(ws, 'charades_r50_lfb_nl.yaml', TINY + ['MODEL.NUM_CLASSES', 157], 64, 8, 2)


def test_full_size_config2_forward_backward(ws):
    """BASELINE.json config 2: R50-I3D-NL + FBO-NL-2L, 2 clips of 32x224x224, R=4, L=300."""
    _train_case(ws, 'ava_r50_lfb_nl.yaml', FULL, 224, 32, 2, check_all_grads=False)


def test_full_size_config1_baseline_forward_test_crop(ws):
    """BASELINE.json config 1: baseline forward (no LFB), test-mode graph."""
    from oracle import model as OM
    ov = FULL + ['TEST.CROP_SIZE', 224]
    H.setup_cfg('ava_r50_baseline.yaml', ov)
    ocfg = H.oracle_cfg('ava_r50_baseline.yaml', ov)
    params = OM.make_params(ocfg, seed=2, split='val')
    inputs = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=2, crop=224, frames=32)
    model, sfx = H.build('val', False)
    H.feed_params(params)
    H.feed_inputs(inputs, sfx)
    ws.RunNet(model.net.Proto().name)
    _, blobs, _ = _oracle(ocfg, params, inputs, 'val', False)
    for b in ['box_pooled', 'pool5', 'pred']:
        e = H.rel(ws.FetchBlob('gpu_0/' + b), blobs[b].detach().numpy())
        print(b, e)
        assert e < FWD_TOL, (b, e)


def _val_lfb_case(ws, yaml_name, overrides, crop, frames, rois_per_clip, fold, runs=1):
    from oracle import model as OM
    from core.config import config as cfg
    from vlfb import executor as X
    H.setup_cfg(yaml_name, overrides)
    cfg.B200.FBO_FOLD = fold
    ocfg = H.oracle_cfg(yaml_name, overrides)
    params = OM.make_params(ocfg, seed=2, split='val')
    inputs = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=rois_per_clip, crop=crop, frames=frames)
    model, sfx = H.build('val', False)
    H.feed_params(params)
    H.feed_inputs(inputs, sfx)
    net = ws.current().nets[model.net.Proto().name]
    assert sum(isinstance(s, X.FboFoldStep) for s in net.steps) == (cfg.FBO_NL.NUM_LAYERS if fold else 0)
    _, blobs, _ = _oracle(ocfg, params, inputs, 'val', False)
    out = {}
    for run in range(runs):                      # runs >= 4: the last ones are CUDA-graph replays
        ws.RunNet(model.net.Proto().name)
        for b in ['lfb_nl0_affinity_prob', 'lfb_nl%d_sum' % (cfg.FBO_NL.NUM_LAYERS - 1), 'pool5', 'pred', 'prob']:
            e = H.rel(ws.FetchBlob('gpu_0/' + b).reshape(-1), blobs[b].detach().numpy().reshape(-1))
            out[b] = e
            assert e < FWD_TOL, (b, e, fold, run)
    print('[%s val fold=%s] %s' % (yaml_name, fold, ' '.join('%s=%.2e' % kv for kv in out.items())))


@pytest.mark.parametrize('fold', [True, False])
def test_tiny_inference_fbo_fold(ws, fold):
    """Test-mode LFB net: every FBO-NL layer is one pass over the raw bank (FboFoldStep) -- and the as-written
    lowering of the same graph -- against the oracle; eager runs and graph replays."""
    _val_lfb_case(ws, 'ava_r50_lfb_nl_3l.yaml', TINY, 64, 8, 3, fold, runs=5)


def test_full_size_inference_with_bank_fold(ws):
    """ava_r50_lfb_nl shapes at inference: 2 clips of 32x224x224, R=4, L=300 bank rows x 2048."""
    _val_lfb_case(ws, 'ava_r50_lfb_nl.yaml', FULL + ['TEST.CROP_SIZE', 224], 224, 32, 2, True)


def test_tiny_r101_3l_train_step(ws):
    """BASELINE.json config 4 architecture (R101-I3D-NL + FBO-NL-3L: 23 res4 blocks, NL at conv4_{6,13,20}), tiny
    clips, tf32 parity mode.  101 layers accumulate more TF32 rounding (and more ReLU / arg-max flips, see the module
    docstring) than 50: measured median relative L2 of the gradients 2.0e-2 (worst tensor conv1_w 8.0e-2, min cosine 0.9968), so the median bound is
    3e-2 here; the per-tensor bounds (L2 <= 0.15, cosine >= 0.98) and the 1e-3 forward bound are unchanged."""
    _train_case(ws, 'ava_r101_lfb_nl_3l.yaml', TINY, 64, 8, 2, median_tol=3e-2)


def test_sgd_step_and_determinism_of_forward(ws):
    from oracle import ops as O
    from core.config import config as cfg
    model, params, p64 = _train_case(ws, 'ava_r50_lfb_nl.yaml', TINY, 64, 8, 2)
    a = ws.FetchBlob('gpu_0/pred').copy()
    model.UpdateWorkspaceLr(10)
    lr = float(ws.FetchBlob('gpu_0/lr'))
    ws.RunNet(model.net.Proto().name)
    for name in ['pred_w', 'res5_2_branch2c_w', 'lfb_1x1_w']:
        # the fused update must be exact given the GPU's own gradient of the previous run
        g_gpu = torch.tensor(ws.FetchBlob('gpu_0/' + name + '_grad')).double()
        p_ref, _ = O.nesterov_update(params[name].double(), p64[name].grad, torch.zeros_like(p64[name]), lr,
                                     cfg.SOLVER.MOMENTUM, cfg.SOLVER.WEIGHT_DECAY)
        step_ref = (p_ref.detach() - params[name].double()).numpy()
        step_gpu = ws.FetchBlob('gpu_0/' + name).astype(np.float64) - params[name].double().numpy()
        assert np.linalg.norm(step_gpu - step_ref) / np.linalg.norm(step_ref) < 0.15, name
    assert np.array_equal(ws.FetchBlob('gpu_0/res2_0_branch2a_bn_s'), params['res2_0_branch2a_bn_s'].numpy())
    assert not np.array_equal(a, 0 * a)


def test_graph_replay_rebinds_its_blobs_after_another_net_ran(ws):
    """ws.blobs is shared by all nets.  Net A (train) is captured; net B (the test net on other inputs) then runs and
    rebinds 'pred', 'pool5', 'box_pooled', ...; a replay of A must hand FetchBlob ITS tensors again.  Also: a second
    input signature (another RoI count) gets its own cached graph instead of evicting the first."""
    from oracle import model as OM
    H.setup_cfg('ava_r50_lfb_nl.yaml', TINY)
    ocfg = H.oracle_cfg('ava_r50_lfb_nl.yaml', TINY)
    params = OM.make_params(ocfg, seed=2)
    model_a, sfx_a = H.build('train', True)
    model_b, sfx_b = H.build('test', False)
    H.feed_params(params)
    name_a, name_b = model_a.net.Proto().name, model_b.net.Proto().name
    net_a = ws.current().nets[name_a]
    net_a.update_ops = []                                   # keep the weights fixed: every run of A is the same function
    in_a = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=2, crop=64, frames=8, seed=70)
    in_a2 = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=3, crop=64, frames=8, seed=71)
    in_b = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=2, crop=64, frames=8, seed=72)
    H.feed_inputs(in_a, sfx_a)
    ws.RunNet(name_a)
    torch.cuda.synchronize()
    want = dict((n, ws.FetchBlob('gpu_0/' + n).copy()) for n in ('pred', 'pool5', 'box_pooled', 'loss'))
    for _ in range(3):
        ws.RunNet(name_a)
    assert len(net_a._graphs) == 1
    H.feed_inputs(in_b, sfx_b)
    ws.RunNet(name_b)                                       # rebinds the shared output names
    torch.cuda.synchronize()
    other = ws.FetchBlob('gpu_0/pred').copy()
    H.feed_inputs(in_a, sfx_a)
    ws.RunNet(name_a)                                       # replay of the captured step
    torch.cuda.synchronize()
    for n, v in want.items():
        got = ws.FetchBlob('gpu_0/' + n)
        assert np.allclose(got, v, rtol=1e-5, atol=1e-6), n
    assert not np.allclose(other, want['pred'], rtol=1e-3, atol=1e-5), 'net B should have produced different predictions'
    # a second signature: captured next to the first, both replay correctly afterwards
    H.feed_inputs(in_a2, sfx_a)
    for _ in range(4):
        ws.RunNet(name_a)
    torch.cuda.synchronize()
    assert len(net_a._graphs) == 2
    pred2 = ws.FetchBlob('gpu_0/pred').copy()
    assert pred2.shape[0] == 6
    H.feed_inputs(in_a, sfx_a)
    ws.RunNet(name_a)
    torch.cuda.synchronize()
    assert np.allclose(ws.FetchBlob('gpu_0/pred'), want['pred'], rtol=1e-5, atol=1e-6)
    assert len(net_a._graphs) == 2


# ---------------------------------------------------------------------------- full-size configs 3 / 4, other heads, files
def test_full_size_config3_r50_fbo_nl_3l_all_gradients(ws):
    """BASELINE.json config 3 shapes (ava_r50_lfb_nl_3l.yaml): full 32x224x224 train step, EVERY trainable tensor's
    gradient against the fp64 oracle."""
    _train_case(ws, 'ava_r50_lfb_nl_3l.yaml', FULL, 224, 32, 2, check_all_grads=True)


def test_full_size_config4_r101_fbo_nl_3l_tf32(ws):
    """BASELINE.json config 4 architecture (ava_r101_lfb_nl_3l.yaml: res4 = 23 blocks, NL at conv4_{6,13,20}) at full
    size in the tf32 parity mode (the bf16 storage mode of config 4 is not built): 174 trainable tensors."""
    _train_case(ws, 'ava_r101_lfb_nl_3l.yaml', FULL, 224, 32, 2, check_all_grads=True, median_tol=3e-2)


def test_full_size_config2_simt_fp32_engine(ws):
    """The same full-size step on the SIMT fp32 engine (no tensor cores, same rounding points): separates tcgen05 /
    TMA kernel error from the ReLU-flip noise that TF32 rounding of the activations causes in both engines."""
    _train_case(ws, 'ava_r50_lfb_nl.yaml', FULL, 224, 32, 2, backend='simt', check_all_grads=True)


@pytest.mark.parametrize('yaml_name', ['ava_r50_lfb_avg.yaml', 'ava_r50_lfb_max.yaml'])
def test_tiny_fbo_avg_max_heads(ws, yaml_name):
    """SURVEY 8f rank 3: the pooling feature-bank operators (lfb_helper.py:106-127) on the GPU path."""
    _train_case(ws, yaml_name, TINY, 64, 8, 2)


def test_checkpoint_round_trip_through_the_device_param_store(ws, tmp_path):
    """SURVEY 8f rank 2 on the GPU: save_model_params -> fresh workspace -> initialize_params_from_file.  Exercises the
    device layouts a file must survive: conv weights [Cout][kT][kH][kW][Cin], the stem padded to 8 px x 4 ch, the
    TF32 operand copy (Pt) refreshed on load, momentum; the reloaded net must reproduce the step bit for bit.  (The
    original's second step folds gradient sums into dgrad epilogues, the reloaded net's first step cannot: the
    deferred two-term sums, executor.LAZY_GRAD_SUM, would associate a three-term sum differently, so they are off.)"""
    from oracle import model as OM
    from utils import checkpoints as CK
    H.setup_cfg('ava_r50_lfb_nl.yaml', TINY)
    ocfg = H.oracle_cfg('ava_r50_lfb_nl.yaml', TINY)
    params = OM.make_params(ocfg, seed=2)
    inputs = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=2, crop=64, frames=8)
    from vlfb import executor as X
    lazy0, X.LAZY_GRAD_SUM = X.LAZY_GRAD_SUM, False
    try:
        _checkpoint_round_trip(ws, tmp_path, ocfg, params, inputs, CK)
    finally:
        X.LAZY_GRAD_SUM = lazy0


def _checkpoint_round_trip(ws, tmp_path, ocfg, params, inputs, CK):
    import pickle
    model, sfx = H.build('train', True)
    H.feed_params(params)
    H.feed_inputs(inputs, sfx)
    model.UpdateWorkspaceLr(10)
    name = model.net.Proto().name
    ws.RunNet(name)                                         # one SGD step: weights moved, momentum non-zero
    torch.cuda.synchronize()
    path = os.path.join(str(tmp_path), 'c2_model_iter1.pkl')
    CK.save_model_params(model, path, 0)
    with open(path, 'rb') as f:
        saved = pickle.load(f)['blobs']
    assert saved['conv1_w'].shape == (64, 3, 5, 7, 7) and saved['res4_0_branch2a_w'].shape == (256, 512, 3, 1, 1)
    assert np.abs(saved['conv1_w'] - params['conv1_w'].numpy()).max() > 0
    ws.RunNet(name)                                         # the step the reloaded model must reproduce
    torch.cuda.synchronize()
    names = ['conv1_w', 'res3_1_branch2b_w', 'nonlocal_conv4_1_theta_w', 'lfb_nl1_out_w', 'pred_w', 'pred_b']
    want = dict((k, ws.FetchBlob('gpu_0/' + k).copy()) for k in names + [n + '_momentum' for n in names])
    want_loss = float(ws.FetchBlob('gpu_0/loss'))
    H.setup_cfg('ava_r50_lfb_nl.yaml', TINY)
    ws.ResetWorkspace()
    model2, sfx2 = H.build('train', True)
    it, lr = CK.initialize_params_from_file(model2, path)
    assert it == 1
    store = ws.current().params
    stem = store.phys('conv1_w')
    assert tuple(stem.shape) == (64, 5, 7, 8, 4) and float(stem[:, :, :, 7, :].abs().max()) == 0 and float(stem[..., 3].abs().max()) == 0
    from util import tf32_round
    assert torch.equal(store.tf32('res3_1_branch2b_w').cpu(), tf32_round(store.phys('res3_1_branch2b_w').cpu()))
    H.feed_inputs(inputs, sfx2)
    ws.RunNet(model2.net.Proto().name)
    torch.cuda.synchronize()
    assert float(ws.FetchBlob('gpu_0/loss')) == want_loss
    for k, v in want.items():
        assert np.array_equal(ws.FetchBlob('gpu_0/' + k).view(np.int32), v.view(np.int32)), k
