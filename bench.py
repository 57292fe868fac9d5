#!/usr/bin/env python
"""bench.py -- clips/sec of the LFB hot path (BASELINE.json config 2: R50-I3D-NL + FBO-NL-2L,
forward + backward + SGD, 2 synthetic 32x224x224 clips / 4 RoIs / 300-row bank per GPU).

  python bench.py --gpus N --steps K --warmup W            # this implementation (tcgen05 path)
  python bench.py --impl reference --gpus N --steps K ...  # CPU reference arm (oracle restatement)

One JSON line on stdout (rank 0).  `value` = device-resident throughput (inputs already in HBM, CUDA-graph replay),
`e2e` = through EnqueueBlobs / RunNet / FetchBlob with pinned host buffers (H2D + loss D2H inside the timed region),
`roofline` = the tcgen05 gathered-GEMM kernel (all launches of one step; by_stage / by_kind; DRAM traffic from the tracked
ncu launch list) against the measured tensor peak, `cpu_baseline` = the oracle timed on the host cores, `fbo_microbench` =
bench_fbo.py cases (BASELINE configs[4]), `large_batch` = the same step at 8 clips per GPU (sub-process), `clocks` =
nvidia-smi samples taken while the timed regions ran.  N > 1 (torchrun): max over ranks, weak scaling, the N=1-only extras
are skipped.

--dump-outputs DIR writes what the last device-resident timed step computed (dump_outputs below) as DIR/<blob>.npy;
inputs and initial weights are seeded, so two builds run with the same arguments can be compared file for file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True          # the benchmark writes nothing into the (possibly read-only) source tree

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, 'video-long-term-feature-banks_b200', 'lib'), ROOT, os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

YAML = 'ava_r50_lfb_nl.yaml'           # --config selects another (CONFIGS below)
CLIPS_PER_GPU = 2
ROIS_PER_CLIP = 2
BANK_ROWS = 300
CONFIGS = {'r50_2l': 'ava_r50_lfb_nl.yaml', 'r50_3l': 'ava_r50_lfb_nl_3l.yaml', 'r101_3l': 'ava_r101_lfb_nl_3l.yaml'}
GFLOP_PER_CLIP = {'r50_2l': 1106.0, 'r50_3l': 1106.0, 'r101_3l': 1551.0}      # SURVEY 8(d), backbone fwd+bwd


def ncu_traffic():
    """DRAM bytes per gemm_tc launch from the tracked ncu summary (profiles/ncu_traffic.json, written by
    scripts/summarize_ncu_launches.py).  bench.py cannot run ncu itself; the file names the kernel source it was
    measured on (sha256 of csrc/gemm_tc.cu) and a stale file is reported as such instead of being quoted."""
    import hashlib
    try:
        with open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')) as f:
            rec = json.load(f)
        src = os.path.join(ROOT, 'video-long-term-feature-banks_b200', 'csrc', 'gemm_tc.cu')
        sha = hashlib.sha256(open(src, 'rb').read()).hexdigest()
        if rec.get('gemm_tc_sha256') != sha:
            return None, 'profiles/ncu_traffic.json is stale (measured on another gemm_tc.cu: %s)' % rec.get('commit', '?')
        return float(rec['dram_bytes_per_gemm_launch']), rec.get('source', 'profiles/ncu_traffic.json')
    except Exception as exc:
        return None, 'no tracked ncu summary (%r)' % (exc,)


def fbo_gflop(rois, bank_rows, layers):
    fwd = 2.0 * rois * (2048 * 512 + bank_rows * 2048 * 512 +
                        layers * (2 * 512 ** 2 + 2 * bank_rows * 512 ** 2 + 2 * bank_rows * 512))
    return 3.0 * fwd / 1e9


def stage_of(label):
    """Blob name of a graph step -> stage of the network (the north star quotes res4/res5 separately)."""
    n = label.split('/')[-1]
    if n.startswith('conv1') or n.startswith('res_conv1'):
        return 'conv1'
    for st in ('res2', 'res3', 'res4', 'res5'):
        if n.startswith(st + '_'):
            return st
    if n.startswith('nonlocal_conv3'):
        return 'nl3'
    if n.startswith('nonlocal_conv4'):
        return 'nl4'
    if n.startswith('lfb') or 'fbonl' in n:
        return 'fbo'
    return 'head'


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons while the timed regions run: ONE long-lived `nvidia-smi -lms` process started
    before them and read by this thread (no process is forked inside a timed region; scripts/diag_e2e.py measured the
    end-to-end loop at 12.50 ms with this sampler running and 12.48 ms without, profiles/r02_diag_e2e_call_r.txt)."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index, period_ms=100):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.samples, self.stop_flag, self.proc, self.period_ms = index, [], False, None, period_ms

    def run(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
            for line in self.proc.stdout:                   # blocking read: the GIL is released while waiting
                if self.stop_flag:
                    break
                v = [t.strip() for t in line.decode(errors='replace').split(',')]
                if len(v) >= 6:
                    self.samples.append(v)
        except Exception:
            pass

    def stop(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(s[2 + i] == 'Active' for s in self.samples)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': int(self.samples[0][1]),
                'reasons': reasons, 'samples': len(self.samples)}


DUMP_MAX_ELEMS = 1 << 15       # per dumped tensor: 2 x ~120 trainable tensors stay well under 64 MB of float32
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(workspace, trainable, out_dir):
    """Write what the training step hands its caller after the last timed step, as float32 .npy files named after
    the blobs: `loss`, the logits `pred`, and every trainable parameter after the SGD update (`<param>`) with the
    gradient of that step (`<param>_grad`).  A tensor of more than DUMP_MAX_ELEMS elements is written as a fixed
    sample of its flattened (logical-layout) elements: sorted indices drawn without replacement by a generator seeded
    with the blob name, so the same elements are sampled in every run and every build."""
    import zlib
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    names = ['loss', 'pred'] + trainable + [p + '_grad' for p in trainable]
    total = 0
    for n in names:
        a = np.asarray(workspace.FetchBlob('gpu_0/' + n), dtype=np.float32)
        if a.size > DUMP_MAX_ELEMS:
            rng = np.random.default_rng(zlib.crc32(n.encode()))
            a = a.reshape(-1)[np.sort(rng.choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        total += a.nbytes
        assert total <= DUMP_MAX_BYTES, 'dumped outputs exceed %d bytes' % DUMP_MAX_BYTES
        np.save(os.path.join(out_dir, n + '.npy'), a)


def measured_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return json.load(f), 'measured'
    except Exception:
        return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback'


# ------------------------------------------------------------------------------------ CPU reference arm
def cpu_threads():
    """Threads for the CPU arm.  Measured on the B200 host (profiles/r01_cpu_thread_sweep.txt, 128
    logical cores): 8 -> 3.0 s/clip, 16 -> 2.65, 32 -> 2.95, 64 -> 4.7, 128 -> 95: oneDNN's 3-D
    convolutions stop scaling at 16 threads, so that is what the baseline uses (all cores if fewer)."""
    return min(os.cpu_count() or 1, 16)


def oracle_setup(n_clips, num_gpus):
    import harness as H
    from oracle import model as OM
    ov = ['NUM_GPUS', num_gpus, 'TRAIN.BATCH_SIZE', n_clips * num_gpus, 'TRAIN.DROPOUT_RATE', 0.0]
    ocfg = H.oracle_cfg(YAML, ov)
    params = OM.make_params(ocfg, seed=2)
    for v in params.values():
        v.requires_grad_(True)
    inputs = OM.make_inputs(ocfg, n_clips=n_clips, rois_per_clip=ROIS_PER_CLIP)
    return OM, ocfg, params, inputs


def oracle_step(OM, ocfg, params, inputs, state, lr=1e-4, momentum=0.9):
    """The same step as the GPU arm: forward, backward, weight decay + Nesterov momentum SGD in the Caffe2 form
    (model_builder_video.py:375-388: g += wd p; m' = mu m + lr g; p -= (1 + mu) m' - mu m), frozen affine layers."""
    import torch
    blobs, prob, loss = OM.forward(ocfg, params, inputs, 'train')
    loss.backward()
    wd, wd_bn = float(ocfg['SOLVER']['WEIGHT_DECAY']), float(ocfg['SOLVER']['WEIGHT_DECAY_BN'])
    with torch.no_grad():
        for name, p in params.items():
            if p.grad is not None and not (name.endswith('_bn_s') or name.endswith('_bn_b')):
                g = p.grad.add(p, alpha=wd_bn if '_bn' in name else wd)
                m = state.setdefault(name, torch.zeros_like(p))
                m_new = m.mul(momentum).add_(g, alpha=lr)
                p.sub_(m_new.mul(1.0 + momentum).sub_(m, alpha=momentum))
                state[name] = m_new
            p.grad = None
    return float(loss)


def run_reference(args):
    import torch
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = cpu_threads()
    torch.set_num_threads(cores)
    OM, ocfg, params, inputs = oracle_setup(CLIPS_PER_GPU, 1)
    state = {}
    for _ in range(args.warmup):
        oracle_step(OM, ocfg, params, inputs, state)
    t0 = time.time()
    for _ in range(args.steps):
        oracle_step(OM, ocfg, params, inputs, state)
    dt = (time.time() - t0) / max(args.steps, 1)
    value = CLIPS_PER_GPU / dt
    sample = ('%d clips (32x224x224, R=%d RoIs, L=%d) fwd+bwd+wd+Nesterov SGD per step, oracle restatement on PyTorch-CPU '
              'fp32' % (CLIPS_PER_GPU, CLIPS_PER_GPU * ROIS_PER_CLIP, BANK_ROWS))
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value,
        'unit': 'clips/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(1),
        'cpu_baseline': {'value': value, 'unit': 'clips/s', 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': 'clips/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


METRIC = 'clips/sec (32x224^2) R50-I3D-NL+FBO-NL fwd+bwd'


def workload_config(n_gpus):
    """Identical for both arms (the driver compares them)."""
    return {'workload': '%s: %d clips/GPU 32x224^2, R=%d, L=%d, fwd+bwd+SGD' % (
                YAML.replace('.yaml', ''), CLIPS_PER_GPU, CLIPS_PER_GPU * ROIS_PER_CLIP, BANK_ROWS),
            'clips_per_gpu': CLIPS_PER_GPU, 'parallelism': 'dp%d' % n_gpus}


# ------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import numpy as np
    import torch
    import harness as H
    from core.config import config as cfg
    from oracle import model as OM   # synthetic-input generator only (SURVEY section 8d); never on the timed path
    from vlfb import dist as vdist
    from vlfb import kernels as K
    from vlfb import workspace

    rank, world = vdist.init_from_env()
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    assert world == args.gpus or world == 1, 'launch with torchrun --nproc-per-node %d' % args.gpus
    n_gpus = world

    ov = ['NUM_GPUS', n_gpus, 'TRAIN.BATCH_SIZE', CLIPS_PER_GPU * n_gpus]
    H.setup_cfg(YAML, ov)
    cfg.RNG_SEED = 2                       # identical initial weights on every rank
    cfg.B200.CUDA_GRAPH = not args.no_graph
    workspace.ResetWorkspace()
    model, sfx = H.build('train', True)
    ocfg = H.oracle_cfg(YAML, ov)
    if rank == 0:      # synthetic weights of bounded dynamic range (SURVEY section 8d generator), then broadcast
        H.feed_params(OM.make_params(ocfg, seed=2))
    vdist.install(workspace.current())
    vdist.broadcast_params(workspace.current().params)
    workspace.FeedBlob('gpu_0/lr', np.array(1e-4, dtype=np.float32))    # keeps random-weight training finite

    inputs = OM.make_inputs(ocfg, n_clips=CLIPS_PER_GPU, rois_per_clip=ROIS_PER_CLIP, seed=100 + rank)
    host = dict((k, v.contiguous().pin_memory()) for k, v in inputs.items())
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    name = model.net.Proto().name

    def feed():
        for k, v in host.items():
            workspace.FeedBlob('gpu_0/%s%s' % (k, sfx), v)

    def barrier():
        if n_gpus > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if n_gpus == 1:
            return ms
        t = torch.tensor([ms], device='cuda')
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput: inputs already in HBM
    feed()
    for _ in range(args.warmup):
        workspace.RunNet(name)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)                     # nvidia-smi is up and sampling before the timed regions start
    barrier()
    K.LAUNCHES = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        workspace.RunNet(name)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    launches = K.LAUNCHES // max(args.steps, 1)
    if rank == 0 and args.dump_outputs:  # before the loops below train the weights further
        dump_outputs(workspace, model.TrainableParams(), args.dump_outputs)

    # ---- end to end through the public API: every step's inputs travel host (pinned) -> device inside the timed
    # region and the loss is read back every step.  EnqueueBlobs is the stand-in for the reference's BlobsQueue
    # feeder: the copy of batch i+1 runs on a side stream behind step i, RunNet dequeues it (layout conversion +
    # TF32 rounding) and replays the step, FetchBlob synchronises.
    def enqueue():
        workspace.EnqueueBlobs(dict(('gpu_0/%s%s' % (k, sfx), v) for k, v in host.items()))

    enqueue()
    for _ in range(2):
        workspace.RunNet(name)
        enqueue()
        loss = float(workspace.FetchBlob('gpu_0/loss'))
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        workspace.RunNet(name)          # consumes the queued batch
        enqueue()                       # H2D of the next batch, overlapped with this step
        loss = float(workspace.FetchBlob('gpu_0/loss'))
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3       # the timed region ends HERE (rounds 1 and 2 up to call R read the wall
    workspace.RunNet(name)                           # clock after this drain step: one step in K too many, e2e understated)
    barrier()
    e2e_ms = max_over_ranks(max(e0.elapsed_time(e1), wall_ms)) / args.steps
    e2e_mode = 'FetchBlob(loss) after every RunNet (blocking)'

    # ---- the same loop with the loss read back asynchronously: step i's loss is copied to pinned host memory by
    # FetchBlobAsync right behind step i and collected after step i+1 has been launched, so the host's launch work
    # overlaps the device.  Every step's inputs still travel H2D and every step's loss D2H inside the timed region.
    e2e_async_ms = None
    try:
        enqueue()
        barrier()
        t0 = time.perf_counter()
        e0.record()
        pending = None
        for _ in range(args.steps):
            workspace.RunNet(name)
            enqueue()
            nxt = workspace.FetchBlobAsync('gpu_0/loss')
            if pending is not None:
                loss = float(pending.get())
            pending = nxt
        loss = float(pending.get())
        e1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        workspace.RunNet(name)          # drain the last queued batch
        barrier()
        e2e_async_ms = max_over_ranks(max(e0.elapsed_time(e1), wall_ms)) / args.steps
    except Exception as exc:             # keep the blocking number if the pipelined loop cannot run
        sys.stderr.write('async e2e loop failed: %r\n' % (exc,))
    e2e_blocking_ms = e2e_ms
    if e2e_async_ms is not None and e2e_async_ms < e2e_ms:
        e2e_ms, e2e_mode = e2e_async_ms, 'FetchBlobAsync(loss): step i read back after step i+1 was launched'
    sampler.stop()

    # ---- roofline of the dominant kernel: every tcgen05 GEMM launch of one more (eager) step is recorded and then
    # replayed back to back between CUDA events (device time per launch; kernels.stop_profile)
    workspace.current().force_eager = True
    if not args.no_roofline:
        K.start_profile()
    workspace.RunNet(name)
    recs = K.stop_profile() if not args.no_roofline else []
    workspace.current().force_eager = False
    gemm_ms = sum(r[1] for r in recs)
    by_kind, by_stage = {}, {}
    if rank == 0 and args.dump_gemms:
        with open(args.dump_gemms, 'w') as f:
            for kind, t, fl, nb, lab in sorted(recs, key=lambda r: -r[1]):
                f.write('%8.3f ms %8.1f TFLOP/s %7.0f GB/s  %-28s %s\n' % (
                    t, fl / 1e9 / t if t else 0, nb / 1e6 / t if t else 0, lab.split('/')[-1], kind))
    if rank != 0:
        return
    peaks, peak_src = measured_peaks()
    peak_tf32 = peaks['bf16_tflops_sustained'] / 2.0                  # kind::tf32 issues at half the bf16 rate
    roof_ms = 0.0            # sum over launches of max(flops / tensor peak, algorithmic bytes / HBM peak)
    for kind, t, f, nb, lab in recs:
        t_roof = max(f / (peak_tf32 * 1e9), nb / (peaks['hbm_gbs'] * 1e6))        # ms
        roof_ms += t_roof
        for table, key in ((by_kind, kind.split(' ')[0]), (by_stage, stage_of(lab))):
            a = table.setdefault(key, [0.0, 0.0, 0, 0.0, 0.0])
            a[0] += t
            a[1] += f
            a[2] += 1
            a[3] += nb
            a[4] += t_roof

    def table_json(tb):
        return dict((k, {'ms': round(v[0], 4), 'tflops': round(v[1] / 1e9 / v[0], 1) if v[0] else 0, 'launches': v[2],
                         'tensor_frac': round(v[1] / 1e9 / v[0] / peak_tf32, 3) if v[0] else 0,
                         'alg_gbs': round(v[3] / 1e6 / v[0], 0) if v[0] else 0,
                         'roof_frac': round(v[4] / v[0], 3) if v[0] else 0}) for k, v in sorted(tb.items()))
    assert np.isfinite(loss), 'loss is not finite'
    layers = cfg.FBO_NL.NUM_LAYERS
    rois = CLIPS_PER_GPU * ROIS_PER_CLIP
    gflop_step = CLIPS_PER_GPU * GFLOP_PER_CLIP[args.config] + fbo_gflop(rois, BANK_ROWS, layers)
    achieved = gflop_step / gemm_ms if gemm_ms > 0 else 0.0          # GFLOP/ms == TFLOP/s
    traffic, traffic_src = ncu_traffic()
    clips = CLIPS_PER_GPU * n_gpus

    # ---- CPU baseline: the oracle on this box's host cores, bounded sample (N=1 only)
    cpu = None
    if n_gpus == 1 and not args.no_cpu_baseline:
        cores = cpu_threads()
        torch.set_num_threads(cores)
        OMo, oc, op, oi = oracle_setup(CLIPS_PER_GPU, 1)
        ost = {}
        oracle_step(OMo, oc, op, oi, ost)
        t0 = time.time()
        nrep = 2
        for _ in range(nrep):
            oracle_step(OMo, oc, op, oi, ost)
        cpu = {'value': nrep * CLIPS_PER_GPU / (time.time() - t0), 'unit': 'clips/s', 'cores': cores, 'kind': 'port',
               'sample': '%d timed steps of %d clips (32x224x224, R=%d, L=%d) fwd+bwd+wd+Nesterov SGD, PyTorch-CPU fp32 '
                         'oracle restatement (the Caffe2 reference cannot run here)' % (
                             nrep, CLIPS_PER_GPU, CLIPS_PER_GPU * ROIS_PER_CLIP, BANK_ROWS)}

    # ---- FBO-NL microbenchmark (BASELINE configs[4], bench_fbo.py) on the same box: the training-config bank, a folded
    # inference bank and a large one (HBM-bound scan); resets the workspace, so it runs after everything above
    fbo = None
    if n_gpus == 1 and not args.no_fbo:
        try:
            import bench_fbo
            fbo = []
            for mode, R_, L_ in (('train', rois, BANK_ROWS), ('infer_fold', rois, BANK_ROWS), ('infer_fold', 64, 1200),
                                 ('infer_fold', 256, 3600), ('infer_fold_bf16', 64, 1200), ('infer_fold_bf16', 256, 3600)):
                r = bench_fbo.run_case(mode, R_, L_, 2, 10, 3, peaks)
                fbo.append(dict((k, r[k]) for k in ('mode', 'R', 'L', 'layers', 'ms', 'launches', 'gbs', 'hbm_frac',
                                                    'tflops_as_written', 'scan')))
        except Exception as exc:
            fbo = {'error': repr(exc)}

    # ---- the same step at a larger per-GPU batch (SURVEY 8d config 3: "additionally report best per-GPU batch, e.g. 8"):
    # a separate process (fresh workspace), device-resident timing only; the headline stays the reference's 2 clips / GPU
    large = None
    if n_gpus == 1 and args.large_batch > CLIPS_PER_GPU:
        try:
            cmd = [sys.executable, os.path.abspath(__file__), '--gpus', '1', '--steps', str(args.steps), '--warmup',
                   str(args.warmup), '--config', args.config, '--clips-per-gpu', str(args.large_batch),
                   '--no-cpu-baseline', '--no-fbo', '--large-batch', '0']
            out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
            sub = json.loads(out.stdout.decode().strip().splitlines()[-1])
            large = {'clips_per_gpu': args.large_batch, 'value': sub['value'], 'unit': 'clips/s',
                     'ms_per_step': sub['ms_per_step'], 'e2e': sub['e2e']['value'],
                     'roofline_frac': sub['roofline']['frac'], 'roofline_achieved_tflops': sub['roofline']['achieved'],
                     'tensor_frac_by_stage': dict((k, v['tensor_frac']) for k, v in sub['roofline']['by_stage'].items()),
                     'gpu_launches': sub['gpu_launches'],
                     'what': 'the same training step with %d clips (R=%d RoIs) per GPU: tiles fill the 148 SMs and the '
                             'per-launch fixed costs amortise; not the headline (the reference trains 2 clips / GPU)' % (
                                 args.large_batch, args.large_batch * ROIS_PER_CLIP)}
        except Exception as exc:
            large = {'error': repr(exc)}

    print(json.dumps({
        'metric': METRIC, 'value': clips / (ms / 1e3),
        'unit': 'clips/s', 'n_gpus': n_gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'tf32', 'data': 'synthetic',
        'config': dict(workload_config(n_gpus),
                       l2='activations (>1 GB/step) exceed the 126 MB L2 between launches; no explicit flush',
                       dropout='Philox, enabled', cuda_graph=bool(cfg.B200.CUDA_GRAPH), weights='random-init'),
        'e2e': {'value': clips / (e2e_ms / 1e3), 'unit': 'clips/s', 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': 4, 'ms_per_step': e2e_ms, 'loss_readback': e2e_mode,
                'ms_per_step_blocking_fetch': e2e_blocking_ms, 'ms_per_step_async_fetch': e2e_async_ms},
        'gpu_launches': launches,
        'clocks': sampler.summary(),
        'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': peak_tf32, 'unit': 'TFLOP/s',
                     'frac': achieved / peak_tf32 if peak_tf32 else None, 'traffic': traffic,
                     'traffic_source': traffic_src,
                     'flop_per_launch': gflop_step * 1e9 / max(len(recs), 1),
                     'kernel': 'vlfb::tc::gemm_tc_kernel: all %d launches of one step; device time of each launch = its '
                               'parameter block replayed 5x back to back between two CUDA events on the launching stream '
                               '(no host launch latency in the number): sum %.2f ms; the captured step takes %.2f ms in '
                               'total' % (len(recs), gemm_ms, ms),
                     'peak_source': '%s bf16_tflops_sustained / 2 (kind::tf32)' % peak_src,
                     'per_launch_roofline': {
                         'what': 'sum over the GEMM launches of max(flops / tensor peak, algorithmic bytes / HBM peak) '
                                 '/ measured time: the fp32 activations make the res2/res3/stem layers HBM-bound',
                         'roof_ms': round(roof_ms, 3), 'measured_ms': round(gemm_ms, 3),
                         'frac': round(roof_ms / gemm_ms, 3) if gemm_ms else None,
                         'hbm_peak_gbs': peaks['hbm_gbs']},
                     'by_kind': table_json(by_kind), 'by_stage': table_json(by_stage)},
        'cpu_baseline': cpu,
        'fbo_microbench': fbo,
        'large_batch': large,
        'loss': loss,
    }))


def main():
    global YAML, CLIPS_PER_GPU
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-gemms', default='', help='write the per-launch GEMM table of one step here')
    ap.add_argument('--dump-outputs', default='', metavar='DIR', help='write the outputs of the last timed step as '
                    'DIR/<blob>.npy (loss, pred, updated parameters and their gradients; large tensors sampled)')
    ap.add_argument('--no-graph', action='store_true', help='eager launches (for ncu / debugging)')
    ap.add_argument('--no-fbo', action='store_true', help='skip the FBO-NL microbenchmark cases (bench_fbo.py)')
    ap.add_argument('--no-roofline', action='store_true', help='skip the per-launch replay profile (ncu launch lists)')
    ap.add_argument('--config', default='r50_2l', choices=sorted(CONFIGS), help='r50_2l = BASELINE configs[1] (default), '
                    'r50_3l = configs[2] (ava_r50_lfb_nl_3l.yaml), r101_3l = configs[3] architecture')
    ap.add_argument('--clips-per-gpu', type=int, default=CLIPS_PER_GPU, help='clips per GPU and step (default 2 = the '
                    "reference's TRAIN.BATCH_SIZE 16 on 8 GPUs; larger batches fill the 148 SMs better)")
    ap.add_argument('--large-batch', type=int, default=8, help='also time the step at this many clips per GPU in a '
                    'separate process (N=1 only; 0 = skip)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs dumps the b200 arm')
    YAML = CONFIGS[args.config]
    CLIPS_PER_GPU = args.clips_per_gpu
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)
        from vlfb import dist as vdist
        sys.stdout.flush()
        sys.stderr.flush()
        if not vdist.shutdown():
            os._exit(0)          # the result line is out; never hang the launcher on a communicator teardown


if __name__ == '__main__':
    main()
