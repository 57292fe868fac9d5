"""2-GPU data-parallel test on the real path (SURVEY 8d config 3): one process per GPU, NCCL all-reduce of the flat
gradient buffers, tcgen05 kernels.  After one step the replicas hold bit-identical weights, and they equal the
single-GPU step on the concatenated batch up to the fp32 summation order of the weight gradients (one GEMM over both
clips vs. the all-reduced sum of two).  Skipped on machines with fewer than 2 GPUs."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))

TINY = ['TRAIN.CROP_SIZE', 64, 'TRAIN.VIDEO_LENGTH', 8, 'LFB.WINDOW_SIZE', 4, 'TRAIN.DROPOUT_RATE', 0.0,
        'FBO_NL.INPUT_DROPOUT_ON', False, 'FBO_NL.LFB_DROPOUT_ON', False]
CHECK = ['conv1_w', 'res2_0_branch2a_w', 'res3_1_branch2b_w', 'res5_2_branch2c_w', 'nonlocal_conv4_1_out_w', 'lfb_1x1_w',
         'lfb_nl1_theta_b', 'lfb_nl0_out_w', 'pred_w', 'pred_b']


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _step(rank, world, clips_lo, clips_hi, all_inputs, params, out, steps=2):
    import harness as H
    from vlfb import dist as vdist
    from vlfb import kernels, workspace
    kernels.set_gemm_backend('tcgen05')
    workspace.ResetWorkspace()
    n = clips_hi - clips_lo
    H.setup_cfg('ava_r50_lfb_nl.yaml', TINY + ['NUM_GPUS', world, 'TRAIN.BATCH_SIZE', n * world])
    model, sfx = H.build('train', True)
    if rank == 0:
        H.feed_params(params)
    vdist.install(workspace.current())
    vdist.broadcast_params(workspace.current().params)
    rois = all_inputs['proposals']
    sel = (rois[:, 0] >= clips_lo) & (rois[:, 0] < clips_hi)
    inputs = {'data': all_inputs['data'][clips_lo:clips_hi], 'labels': all_inputs['labels'][sel], 'lfb': all_inputs['lfb'][sel]}
    pr = rois[sel].clone()
    pr[:, 0] -= clips_lo
    inputs['proposals'] = pr
    H.feed_inputs(inputs, sfx)
    model.UpdateWorkspaceLr(10)
    for _ in range(steps):
        workspace.RunNet(model.net.Proto().name)
    torch.cuda.synchronize()
    for name in CHECK:
        out[name] = workspace.FetchBlob('gpu_0/' + name).copy()
    out['loss'] = float(workspace.FetchBlob('gpu_0/loss'))
    workspace.ResetWorkspace()


def _worker(rank, world, port, all_inputs, params, ret):
    sys.path.insert(0, HERE)
    import conftest  # noqa: F401  (sys.path setup)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from core import config as C
    C.reset_cfg()
    from vlfb import dist as vdist
    vdist.init_from_env('nccl')
    out = {}
    _step(rank, world, rank, rank + 1, all_inputs, params, out)
    ret[rank] = out
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
def test_two_gpu_nccl_step_equals_single_gpu_step():
    import harness as H
    from oracle import model as OM
    ocfg = H.oracle_cfg('ava_r50_lfb_nl.yaml', TINY + ['NUM_GPUS', 1, 'TRAIN.BATCH_SIZE', 2])
    params = OM.make_params(ocfg, seed=2)
    all_inputs = OM.make_inputs(ocfg, n_clips=2, rois_per_clip=2, crop=64, frames=8)
    port = _free_port()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, port, all_inputs, params, ret), nprocs=2, join=True)
    r0, r1 = ret[0], ret[1]
    single = {}
    _step(0, 1, 0, 2, all_inputs, params, single)
    print('losses: ranks %.6f + %.6f, single %.6f' % (r0['loss'], r1['loss'], single['loss']))
    assert abs((r0['loss'] + r1['loss']) - single['loss']) < 2e-3 * abs(single['loss'])
    for name in CHECK:
        assert np.array_equal(r0[name], r1[name]), name                      # replicas stay in sync, bit for bit
        moved = np.abs(single[name] - params[name].numpy()).max()
        d = np.abs(r0[name] - single[name]).max()
        print('%-28s |update| %.3e  |2-GPU - 1-GPU| %.3e' % (name, moved, d))
        assert moved > 0 and d < 2e-2 * moved + 1e-7, (name, d, moved)        # == the big-batch step
