#!/usr/bin/env python
"""EfficientDet hot-path throughput on N B200s of one node (BASELINE.json metric and configs).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config d0|d4|d7] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step returned to its caller (rank 0) as .npy files: inputs, weights and
the drop-connect stream are seeded, so two builds run with the same arguments can be compared output for output.

--config d0 (default, BASELINE.json configs[1]/[2], the headline metric): EfficientDet-D0 512x512, bs=32 per GPU.
  A "step" = one pass of the hot path over one synthetic batch: backbone -> BiFPN -> head -> FocalLoss forward, then
  backward to every parameter gradient (optimizer excluded, SURVEY.md 8(d)), train mode exactly as reference
  train.py:100-102 (model.train(), is_training, freeze_bn -> drop-connect active, BN frozen).
--config d4 (configs[3]): EfficientDet-D4 1024x1024 (B4 backbone, W_bifpn 224, D_bifpn 6, utils/config_eff.py),
  bs=4 per GPU, same train step.
--config d7 (configs[4]): EfficientDet-D7 1536x1536 (B6 backbone, W_bifpn 384, D_bifpn 8), bs=1 per GPU, inference
  + decode + NMS at eval.py's thresholds (0.4 / 0.5); N>1 = independent replicas, no collective.

One process per GPU; for the train configs with N>1 the model is wrapped in DistributedDataParallel(
find_unused_parameters=True) and the only collective is DDP's NCCL gradient all-reduce (weak scaling).
Prints ONE JSON line on rank 0.

`--impl reference` times the reference's OWN modules (baseline/_ref, installed unmodified by
baseline/install_ref.sh, three run-time shims in baseline/ref_runner.py) on the box's host cores with all the
threads it can use, on a bounded sample of the same workload; if baseline/_ref did not travel it falls back to
the oracle port (oracle/effdet_oracle.py, pinned bit-exact to the reference by tests/golden/) and says so.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(REPO, 'oracle'))

import torch  # noqa: E402

G_ANN = 8
CONFIGS = {
    'd0': dict(net='efficientdet-d0', K=80, W=64, D=2, size=512, bs=32, mode='train', fwd_gflop=64.09,
               metric='EfficientDet-D0 512x512 images/sec (fwd+bwd)',
               workload='EfficientDet-D0 512x512 K=80 bs=32/GPU train step fwd+bwd (configs[1]; configs[2] when N=8)'),
    'd4': dict(net='efficientdet-d4', K=80, W=224, D=6, size=1024, bs=4, mode='train', fwd_gflop=2 * 227.8,
               metric='EfficientDet-D4 1024x1024 images/sec (fwd+bwd)',
               workload='EfficientDet-D4 1024x1024 K=80 bs=4/GPU train step fwd+bwd (configs[3])'),
    'd7': dict(net='efficientdet-d7', K=80, W=384, D=8, size=1536, bs=1, mode='infer', fwd_gflop=2 * 1077.2,
               metric='EfficientDet-D7 1536x1536 images/sec (inference + NMS)',
               workload='EfficientDet-D7 1536x1536 K=80 bs=1/GPU inference + decode + NMS, threshold 0.4 iou 0.5 '
                        '(configs[4], eval.py:349-352)'),
}


def load_peaks():
    p = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d['hbm_gbs'], bf16_tflops=d['bf16_tflops'], bf16_tflops_sustained=d.get('bf16_tflops_sustained'),
                    source='measured')
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source='fallback')


def measured_traffic(kernel_key):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/), or None."""
    p = os.path.join(REPO, 'profiles', 'r02_ncu_traffic.json')
    if not os.path.exists(p):
        return None
    d = json.load(open(p))
    # the capture is only quoted for the kernel source it was taken from
    import hashlib
    csrc = os.path.join(REPO, 'efficientdet.pytorch_b200', 'csrc')
    try:
        h = hashlib.sha1(open(os.path.join(csrc, 'conv_planes.cu'), 'rb').read() + open(os.path.join(csrc, 'tc_ptx.cuh'), 'rb').read()).hexdigest()
    except OSError:
        return None
    if d.get('source_sha1 (conv_planes.cu + tc_ptx.cuh)') != h:
        return None
    return d.get(kernel_key)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(',')]
                if len(f) >= 7:
                    self.rows.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith('active') for r in self.rows)]
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None,
                    sm_max_mhz=float(self.rows[0][1]) if self.rows else None, reasons=reasons, samples=len(self.rows))


def usable_cores():
    """host threads this process may really use: affinity mask, then the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
        if quota != 'max':
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, min(n, 64))


def synthetic(cfgd, B, seed):
    import effdet_oracle as O
    return O.synthetic_batch(B, size=cfgd['size'], G=G_ANN, num_classes=cfgd['K'], seed=seed)


DUMP_BYTES = 60 << 20          # data of all dumped arrays together; with the .npy headers the dump stays under 64 MB


def dump_outputs(outputs, path):
    """Write each named tensor of `outputs` as <path>/<name>.npy: float32, or float64 for integer tensors (exact).
    When they exceed DUMP_BYTES together, every tensor is cut to the same fraction of its elements, at sorted indices
    drawn by a generator seeded with 0, so two runs or two builds with the same arguments store the same elements."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    outputs = {k: v.detach() for k, v in outputs.items() if v is not None}
    total = sum(v.numel() * (4 if v.is_floating_point() else 8) for v in outputs.values())
    frac = min(1.0, DUMP_BYTES / max(total, 1))
    for name, t in outputs.items():
        if frac < 1.0:
            n = max(1, int(t.numel() * frac))
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:n].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        a = t.cpu().numpy()
        np.save(os.path.join(path, name + '.npy'), a.astype(np.float32 if t.is_floating_point() else np.float64))


# ------------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation on the host cores
# ------------------------------------------------------------------------------------------------------------------

def oracle_port_train_steps(cfgd, bs, steps, warmup):
    import effdet_oracle as O
    cfg = O.make_config(cfgd['net'], cfgd['K'], cfgd['W'], cfgd['D'])
    sd = O.init_state_dict(cfg, seed=0)
    sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and 'running' not in k else v) for k, v in sd.items()}
    images, ann = synthetic(cfgd, bs, 0)
    nskip = sum(1 for i, b in enumerate(cfg['blocks']) if b['skip'] and i > 0)

    def step():
        for v in sdg.values():
            if v.is_floating_point():
                v.grad = None
        keeps = [torch.rand([bs, 1, 1, 1]) for _ in range(nskip)]          # train mode: drop-connect active
        cl, rl = O.train_forward(sdg, images, ann, cfg, keep_samples=keeps)
        (cl.mean() + rl.mean()).backward()
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return (time.perf_counter() - t0) / max(steps, 1)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import effdet_oracle as O
    cfgd = CONFIGS[args.config]
    cores = usable_cores()
    torch.set_num_threads(cores)
    sys.path.insert(0, os.path.join(REPO, 'baseline'))
    import ref_runner
    real = ref_runner.available()
    cfg = O.make_config(cfgd['net'], cfgd['K'], cfgd['W'], cfgd['D'])
    sd = O.init_state_dict(cfg, seed=0)
    build = ref_runner.load() if real else None
    detections = None
    if cfgd['mode'] == 'train':
        def timed(bs, steps, warmup):
            images, ann = synthetic(cfgd, bs, 0)
            if real:
                return ref_runner.train_steps(build, cfgd['net'], cfgd['K'], cfgd['W'], cfgd['D'], sd, images, ann, steps, warmup)
            return oracle_port_train_steps(cfgd, bs, steps, warmup)
        bs = args.cpu_bs
        if not bs:
            # bounded sample: pick the per-step batch so that (steps+warmup) steps stay within ~150 s
            t1 = timed(1, 1, 1)
            budget = 150.0 / max(args.steps + args.warmup, 1)
            bs = 1
            for cand in (2, 4, 8):
                if cand <= cfgd['bs'] and t1 * cand * 0.8 <= budget:
                    bs = cand
        dt = timed(bs, args.steps, args.warmup)
    else:
        bs = 1
        images, _ = synthetic(cfgd, 1, 0)
        if real:
            dt, detections = ref_runner.infer_steps(build, cfgd['net'], cfgd['K'], cfgd['W'], cfgd['D'], sd, images, args.steps,
                                                    args.warmup, threshold=args.threshold)
        else:
            with torch.no_grad():
                for _ in range(args.warmup):
                    O.detect(sd, images, cfg, threshold=args.threshold, iou_threshold=0.5)
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    out = O.detect(sd, images, cfg, threshold=args.threshold, iou_threshold=0.5)
                dt = (time.perf_counter() - t0) / max(args.steps, 1)
                detections = int(out[0].numel())
    ips = bs / dt
    kind = 'reference' if real else 'port'
    what = ('the reference\'s own models/ (baseline/_ref, unmodified, torch CPU fp32 + torchvision NMS)' if real else
            'oracle port of the reference (torch CPU fp32); baseline/_ref did not travel')
    sample = '%s, %s of bs=%d per step, %d threads' % (what, 'train step' if cfgd['mode'] == 'train' else 'inference', bs, cores)
    line = dict(metric=cfgd['metric'], value=ips, unit='img/s', n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=dt * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32',
                data='synthetic', impl='reference',
                config=dict(workload=cfgd['workload'] + ' [CPU sample bs=%d]' % bs, global_batch=bs, parallelism='cpu',
                            detections=detections),
                cpu_baseline=dict(value=ips, unit='img/s', cores=cores, kind=kind, sample=sample),
                e2e=dict(value=ips, unit='img/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


def cpu_baseline_subprocess(config, steps, warmup, bs, threshold):
    """the in-line cpu_baseline leg: the reference arm in a child process (it imports the reference's `models`
    package, whose name the product shares), at N=1 only"""
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--config', config, '--steps', str(steps),
           '--warmup', str(warmup), '--cpu-bs', str(bs), '--threshold', str(threshold)]
    env = dict(os.environ)
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK'):
        env.pop(k, None)
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env).stdout.strip().splitlines()
        d = json.loads(out[-1])
        cb = d['cpu_baseline']
        cb['value'] = round(cb['value'], 3)
        cb['sample'] += ', %d timed steps after %d warm-up' % (steps, warmup)
        return cb
    except Exception as e:                                       # the baseline is a reported number, never a blocker
        return dict(value=None, unit='img/s', cores=usable_cores(), kind='unavailable', sample='cpu leg failed: %r' % (e,))


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------

def run_ours(args):
    sys.path.insert(0, os.path.join(REPO, 'efficientdet.pytorch_b200'))
    import torch.distributed as dist
    from models import EfficientDet, _native, _ops
    import effdet_oracle as O

    cfgd = CONFIGS[args.config]
    train = cfgd['mode'] == 'train'
    BS = cfgd['bs']
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert world == args.gpus, 'WORLD_SIZE=%d but --gpus %d (launch with torch.distributed.run)' % (world, args.gpus)
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    # N > 1: the DDP step (NCCL all-reduces included) is replayed as one CUDA graph too -- torch's recipe needs the
    # watchdog's async error handling off before the process group exists (EFFDET_DDP_GRAPH=0: eager DDP; verified on 2 and 8 B200s)
    ddp_graph = train and world > 1 and not args.no_graph and os.environ.get('EFFDET_DDP_GRAPH', '1') != '0'
    if ddp_graph:
        os.environ['TORCH_NCCL_ASYNC_ERROR_HANDLING'] = '0'
        os.environ['NCCL_ASYNC_ERROR_HANDLING'] = '0'
    if world > 1:
        import datetime
        dist.init_process_group(backend='nccl', device_id=dev, timeout=datetime.timedelta(seconds=180))
    _native.load()

    cfg = O.make_config(cfgd['net'], cfgd['K'], cfgd['W'], cfgd['D'])
    model = EfficientDet(num_classes=cfgd['K'], network=cfgd['net'], D_bifpn=cfgd['D'], W_bifpn=cfgd['W'], is_training=train,
                         threshold=args.threshold, iou_threshold=0.5)
    model.load_state_dict(O.init_state_dict(cfg, seed=0))      # well-conditioned random init, same on every rank
    model = model.to(dev)
    if train:
        model.train()
        model.is_training = True
        model.freeze_bn()
    else:
        model.eval()
    net = model
    if world > 1 and train:
        # reference train.py:250 wraps with find_unused_parameters=True (5 dead backbone parameters); the set of
        # unused parameters never changes, so static_graph lets DDP learn it once instead of searching the autograd
        # graph and synchronising a usage bitmap every iteration (EFFDET_DDP_STATIC=0 restores the per-step search)
        static = os.environ.get('EFFDET_DDP_STATIC', '1') != '0'
        side = torch.cuda.Stream(device=dev)          # constructed on a side stream: DDP's AccumulateGrad hooks must not
        side.wait_stream(torch.cuda.current_stream(dev))   # be tied to the legacy stream if the step is to be captured
        with torch.cuda.stream(side):
            net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], find_unused_parameters=True,
                                                            static_graph=static, gradient_as_bucket_view=True,
                                                            bucket_cap_mb=float(os.environ.get('EFFDET_DDP_BUCKET_MB', '25')),
                                                            # BN statistics are frozen (freeze_bn): nothing to re-broadcast per step
                                                            broadcast_buffers=os.environ.get('EFFDET_DDP_BCAST', '0') == '1')
        torch.cuda.current_stream(dev).wait_stream(side)

    torch.manual_seed(0)               # drop-connect masks: the same random stream on every run with the same arguments
    images_h, ann_h = synthetic(cfgd, BS, seed=1000 + rank)
    images_h, ann_h = images_h.pin_memory(), ann_h.pin_memory()
    images_d, ann_d = images_h.to(dev), ann_h.to(dev)
    last = {}

    if train:
        def step(x, a, module=None):
            for p in model.parameters():
                p.grad = None
            cl, rl = (module or net)([x, a])
            loss = cl.mean() + rl.mean()
            loss.backward()
            return loss.detach()
    else:
        def step(x, a, module=None):
            with torch.no_grad():
                det = model(x)
            last['det'] = det
            return det

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    if not ddp_graph:                  # (the DDP graph path warms up on GraphedTrainStep's side stream instead)
        for _ in range(args.warmup):
            step(images_d, ann_d)
    # single-GPU training configs replay the step as ONE CUDA graph (models/graph_step.py: the public helper a user
    # of the drop-in would call): ~480 launches cost the host one cudaGraphLaunch instead of 12-16 ms of Python
    graphed, graph_note, graph_launches = None, 'eager', None
    if train and not args.no_graph and (world == 1 or ddp_graph):
        try:
            from models.graph_step import GraphedTrainStep
            if ddp_graph:
                graphed = GraphedTrainStep(net, images_d, ann_d, warmup=max(11, args.warmup))
                graph_launches = graphed.library_launches
                graph_note = 'cuda graph incl. the NCCL all-reduces (GraphedTrainStep over DDP), %d library kernels per replay' % graph_launches
            else:
                graphed = GraphedTrainStep(model, images_d, ann_d, warmup=0)
                graph_launches = graphed.library_launches        # kernels of this library recorded into the graph
                graph_note = 'cuda graph (GraphedTrainStep), %d library kernels per replay' % graph_launches
            eager_step = step

            def step(x, a, module=None):                     # noqa: F811
                if module is not None:
                    return eager_step(x, a, module)
                return graphed(x, a)
            for _ in range(2):
                step(images_d, ann_d)
        except Exception as e:                               # never let the optimisation block the measurement
            graphed, graph_note = None, 'eager (graph capture failed: %r)' % (e,)
    sampler = ClockSampler(local)
    if rank == 0:                      # one nvidia-smi poller per job, on rank 0's GPU
        sampler.start()
    _native.reset_launch_count()
    ms = timed(lambda: last.__setitem__('out', step(images_d, ann_d)), args.steps)
    launches = graph_launches if graphed is not None else _native.launch_count() // max(args.steps, 1)
    if args.dump_outputs and rank == 0:
        # what a caller of the timed step receives from its last step, before any later step overwrites it: the loss
        # and every parameter gradient (train), or the detections of image 0 (inference)
        if train:
            outs = {'loss': last['out']}
            outs.update(('grad.' + k, p.grad) for k, p in model.named_parameters())
        else:
            outs = dict(zip(('scores', 'classes', 'boxes'), last['out']))
        dump_outputs(outs, args.dump_outputs)

    # host-side issue time of one step (queue empty before, no sync after): how far the CPU runs ahead of the GPU
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    step(images_d, ann_d)
    host_ms = (time.perf_counter() - t0) * 1e3
    torch.cuda.synchronize()

    # end-to-end through the public API with HOST inputs: every step's images + annotations are copied from pinned
    # host memory (double-buffered on a copy stream, i.e. the copy of step i+1 overlaps the compute of step i, like a
    # DataLoader with pin_memory + non_blocking) and every step's result (loss / detections) is read back to the host.
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [(torch.empty_like(images_d), torch.empty_like(ann_d)) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    state = {'i': 0, 'primed': False, 'd2h': 4}

    def h2d(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])
            bufs[slot][0].copy_(images_h, non_blocking=True)
            if train:
                bufs[slot][1].copy_(ann_h, non_blocking=True)
            ready[slot].record(copy_stream)

    def e2e_step():
        i = state['i']
        slot = i & 1
        if not state['primed']:
            h2d(slot)
            state['primed'] = True
        h2d(slot ^ 1)                                   # inputs of the NEXT step go in flight now
        torch.cuda.current_stream().wait_event(ready[slot])
        out = step(bufs[slot][0], bufs[slot][1])
        consumed[slot].record()
        state['i'] = i + 1
        if train:
            return float(out.item())                    # D2H read of the step's result
        host = [t.cpu() for t in out]                   # eval.py:102-104: scores, labels, boxes to the host
        state['d2h'] = sum(t.numel() * t.element_size() for t in host)
        return host

    for ev in consumed:
        ev.record()
    e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    sampler.stop_flag = True
    if rank == 0:
        sampler.join(timeout=2)

    # per-kernel breakdown with CUDA events around every C-ABI launch (extra profiled steps, rank 0)
    roofline, breakdown, cpu_base, kroof = None, None, None, None
    if rank == 0:
        peaks = load_peaks()
        prof = _native.Profiler()
        _native.PROFILER = prof
        psteps = 2
        for _ in range(psteps):
            step(images_d, ann_d, module=model)      # rank-local: no collective outside the timed region
        torch.cuda.synchronize()
        _native.PROFILER = None
        table = prof.table()
        kroof = prof.rooflines(peaks['hbm_gbs'], peaks['bf16_tflops_sustained'] or peaks['bf16_tflops'])
        tot = sum(v[0] for v in table.values())
        breakdown = {k: dict(ms_per_step=round(v[0] / psteps, 4), launches_per_step=v[1] // psteps,
                             share=round(v[0] / tot, 4)) for k, v in sorted(table.items(), key=lambda kv: -kv[1][0])[:(400 if args.full_breakdown else 12)]}
        # dominant kernel class: the dense 3x3 implicit-GEMM conv of head + neck (forward and data-gradient
        # launches of conv_tc_kernel / conv_igemm_kernel).  Algorithmic FLOPs = 2*M*9*Cin*Cout per launch
        # (SURVEY.md 8(d)), summed over the launches of the profiled steps, over their summed device time
        # (CUDA events on the launching stream around every C-ABI call).
        fl, t_ms, n = prof.conv_flops(lambda tag: tag[5] == 3 and tag[3] >= 36 and tag[4] >= 36)
        ach = fl / (t_ms * 1e-3) / 1e12 if t_ms else 0.0
        tc = _ops.tc_enabled()
        peak = peaks['bf16_tflops_sustained'] or peaks['bf16_tflops']
        roofline = dict(kernel=('conv_planes_kernel: TMA-fed tcgen05 bf16x3 implicit GEMM on bf16 hi/lo planes (3 kind::f16 MMAs per '
                                'product, fp32 accum in TMEM), dense 3x3 convs of head+neck, fwd+dgrad' if tc else
                                'conv_igemm_kernel: exact fp32 on the CUDA cores, dense 3x3 convs of head+neck, fwd+dgrad'),
                        bound='tensor', achieved=round(ach, 2), peak=peak, unit='TFLOP/s', frac=round(ach / peak, 4),
                        peak_source=peaks['source'] + ' bf16 cuBLAS, sustained figure (kernel timed inside a long step)',
                        note=('achieved counts ALGORITHMIC fp32-equivalent FLOPs; the tensor pipe executes 3x that '
                              '(bf16 hi/lo split for <=1e-3 parity): tensor-pipe work = %.0f TFLOP/s = %.2f of peak'
                              % (3 * ach, 3 * ach / peak)) if tc else None,
                        launches_per_step=n // psteps, ms_per_step=round(t_ms / psteps, 3),
                        traffic=measured_traffic('conv_planes_kernel<256> 256->256') if (tc and args.config == 'd0') else None)
        if not args.no_cpu and world == 1:      # the CPU leg is an N=1 measurement (the host cores are shared by all ranks)
            if train:
                cpu_base = cpu_baseline_subprocess(args.config, 5 if args.config == 'd0' else 1, 1, 8 if args.config == 'd0' else 1,
                                                   args.threshold)
            else:
                cpu_base = cpu_baseline_subprocess(args.config, 1, 0, 1, args.threshold)

    if rank == 0:
        imgs = BS * world * args.steps
        h2d_bytes = images_h.numel() * 4 + (ann_h.numel() * 4 if train else 0)
        config = dict(workload=cfgd['workload'], global_batch=BS * world,
                      parallelism=('dp%d' % world) if train else ('replicas%d' % world),
                      l2=('per-step working set (GBs of activations) >> 126 MB L2; no explicit flush'),
                      weights='well-conditioned random init (oracle seed 0)',
                      precision=('fp32 storage + fp32 accumulation; 1x1/3x3 convs on tcgen05 with bf16 hi/lo split '
                                 'operands (3 MMAs per product, ~2^-16 per product)') if _ops.tc_enabled()
                      else 'exact fp32 on the CUDA cores')
        if train:
            config['drop_connect'] = 'active (train mode)'
            config['execution'] = graph_note
        else:
            det = last.get('det')
            config.update(threshold=args.threshold, iou_threshold=0.5, detections=int(det[0].numel()) if det is not None else None)
        line = dict(impl='ours', metric=cfgd['metric'], value=round(imgs / (ms * 1e-3), 2), unit='img/s', n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=round(ms / args.steps, 3), higher_is_better=True, scaling='weak',
                    vs_baseline=None, dtype='f32', data='synthetic', config=config,
                    clocks=sampler.summary(),
                    e2e=dict(value=round(imgs / (ms_e2e * 1e-3), 2), unit='img/s',
                             h2d_bytes_per_step=h2d_bytes, d2h_bytes_per_step=state['d2h']),
                    gpu_launches=launches, host_issue_ms_per_step=round(host_ms, 2), roofline=roofline, cpu_baseline=cpu_base, kernel_breakdown=breakdown,
                    kernel_rooflines=kroof if args.full_breakdown else None,
                    model_tflops=round((3 if train else 1) * cfgd['fwd_gflop'] * imgs / (ms * 1e-3) / 1e3, 2))
        print(json.dumps(line), flush=True)
    if world > 1:
        if graphed is not None:
            # with a live CUDA graph that holds NCCL kernels the teardown (graph / communicator destructors) waits
            # forever on this stack (seen on 2 x B200): the result is out, leave without it
            torch.cuda.synchronize()
            dist.barrier(device_ids=[local])
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='d0', choices=sorted(CONFIGS))
    ap.add_argument('--threshold', type=float, default=0.4, help='score threshold of the inference config (eval.py:349 uses 0.4)')
    ap.add_argument('--cpu-bs', type=int, default=0, help='reference arm: images per CPU step (0 = pick a bounded sample)')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg (profiling runs)')
    ap.add_argument('--no-graph', action='store_true', help='issue every launch from Python instead of replaying a CUDA graph')
    ap.add_argument('--full-breakdown', action='store_true', help='list every kernel class in kernel_breakdown')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps write what the last one computed '
                    '(loss and parameter gradients, or detections) as DIR/<name>.npy, at most 64 MB in all')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
