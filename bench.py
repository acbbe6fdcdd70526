#!/usr/bin/env python
"""bench.py — training scans/sec of the mv-3ddet hot path (BASELINE.json config C2: ResNet-50/16 + MinkResNet34,
20 views 480x640, 100k points, bf16) on N B200s of one node, data-parallel over scans.

  python bench.py --gpus 1 --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                      (the CPU port of the reference path on the host cores)

  python bench.py --variant C5|C3|C4 ...                    (the sibling configurations of BASELINE.json; C2 is the headline)
  python bench.py --dump-outputs DIR ...                    (also write the last timed step's outputs as DIR/*.npy)

One JSON line on rank 0. `value`: device-resident inputs, fwd + loss + bwd + grad all-reduce + clip + AdamW, timed with
CUDA events, max over ranks. `e2e`: the same step through model.train_step with pinned HOST inputs (H2D inside the timed
region, loss read back). `roofline`: the sparse-conv gather/GEMM/scatter kernels, algorithmic bytes (pair model,
BASELINE.md §3) / CUDA-event time of each launch, taken in a SEPARATE pass over the same K steps (a CUDA-event pair around
every conv launch, 2D/3D stream overlap off so each kernel is timed alone; kept out of `value` because ~1.7k event pairs per
step cost host time in a host-bound step). `cpu_baseline`: oracle port on host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# The step allocates hundreds of tensors whose sizes follow the data (row counts of the sparse maps differ per batch): with the
# default segment allocator a fragmented pool answers with cudaFree + cudaMalloc cycles (100-400 ms stalls every few steps).
os.environ.setdefault('PYTORCH_CUDA_ALLOC_CONF', 'expandable_segments:True')

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = 'training scans/sec mv-3ddet 20-view (ResNet-50/16 + MinkResNet34, 480x640, 100k pts)'
UNIT = 'scans/s'
# BASELINE.json configs: C2 = the configuration the metric is quoted on; the others are the sibling workloads
VARIANTS = {
    'C2': dict(batch=4, views=20, height=480, width=640, points=100000, kind='det', metric=METRIC,
               model='ResNet-50/16 + MinkResNet34 + FCAF3DHeadRotMat'),
    'C5': dict(batch=4, views=50, height=480, width=640, points=200000, kind='det',
               metric='training scans/sec mv-3ddet 50-view stress (ResNet-50/16 + MinkResNet34, 480x640, 200k pts)',
               model='ResNet-50/16 + MinkResNet34 + FCAF3DHeadRotMat'),
    'C3': dict(batch=1, views=20, height=480, width=640, points=100000, kind='occ',
               metric='training scans/sec occupancy DenseFusionOccPredictor 20-view, 40x40x16 grid',
               model='ResNet-50 + FPN + MinkResNet34 + IndoorImVoxelNeck + ImVoxelOccHead'),
    'C4': dict(batch=12, views=20, height=480, width=480, points=100000, kind='ground',
               metric='training scans/sec mv-grounding SparseFeatureFusion3DGrounder 20-view',
               model='ResNet-50/16 + MinkResNet34 + MinkNeck + text encoder + 6-layer decoder + GroundingHead'),
}


_T0 = time.time()


def log(msg):
    if int(os.environ.get('RANK', 0)) == 0:
        print(f'[bench +{time.time() - _T0:6.1f}s] {msg}', file=sys.stderr, flush=True)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='esb200', choices=['esb200', 'reference'])
    ap.add_argument('--batch', type=int, default=None, help='scans per GPU per step (default by variant; C2: cfg :181 batch_size=4)')
    ap.add_argument('--views', type=int, default=None)
    ap.add_argument('--height', type=int, default=None)
    ap.add_argument('--width', type=int, default=None)
    ap.add_argument('--points', type=int, default=None)
    ap.add_argument('--variant', default='C2', choices=sorted(VARIANTS))
    ap.add_argument('--dtype', default='bf16', choices=['bf16', 'fp32'])
    ap.add_argument('--run-ahead', type=int, default=int(os.environ.get('ESB200_RUN_AHEAD', '1')),
                    help='optimiser steps the host may queue ahead of the device (engine.OptimWrapper.max_run_ahead)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--torch-profile', default='', help='write a torch.profiler kernel table of 2 steps to this path')
    ap.add_argument('--row-order', default=None, choices=['input', 'morton'],
                    help='row order of the sparse tensors (default: ESB200_ROW_ORDER or input); morton = Z-ordered rows')
    ap.add_argument('--dump-outputs', default='', metavar='DIR',
                    help='after the timed steps, write what the last timed step computed as DIR/<name>.npy (dump_outputs)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs records the timed esb200 path; the reference arm times a different step')
    for k, v in VARIANTS[args.variant].items():
        if k in ('batch', 'views', 'height', 'width', 'points') and getattr(args, k) is None:
            setattr(args, k, v)
    return args


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


class ClockSampler:
    """SM clock + throttle reasons sampled through NVML from the MAIN thread (before, twice during and after the timed
    region). A background sampling thread (or spawning nvidia-smi) measurably slows a host-bound step."""

    def __init__(self, index):
        self.index, self.sm, self.reasons_seen, self.max_mhz, self.nv = index, [], set(), None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            phys = index
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            if vis:
                try:
                    phys = int(vis.split(',')[index])
                except Exception:
                    phys = index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
        except Exception:
            self.nv = None

    def sample(self):
        try:
            if self.nv is not None:
                nv = self.nv
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for name, bit in (('hw_slowdown', 0x8), ('sw_thermal_slowdown', 0x20), ('hw_thermal_slowdown', 0x40),
                                  ('sw_power_cap', 0x4)):
                    if r & bit:
                        self.reasons_seen.add(name)
            else:
                out = subprocess.run(['nvidia-smi', f'--id={self.index}', '--query-gpu=clocks.sm,clocks.max.sm',
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True,
                                     timeout=5).stdout.strip().split(',')
                self.sm.append(float(out[0]))
                self.max_mhz = float(out[1])
        except Exception:
            pass

    def summary(self):
        if not self.sm:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': ['unavailable']}
        sm = sorted(self.sm)
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons_seen),
                'samples': len(sm), 'source': 'nvml' if self.nv is not None else 'nvidia-smi'}


class InitialState:
    """The seeded weights and buffers (BatchNorm statistics) a run starts from. fp32 atomics make the training trajectory
    differ from run to run in the last bits, and AdamW and the head's top-k selections amplify that over tens of steps;
    putting this state back before the step whose outputs are dumped gives that step's forward pass identical inputs in
    every run. Restoring is a few launches, enqueued between two steps."""

    def __init__(self, model, arena):
        self.arena = arena
        self.flat = arena.flat.clone()
        self.bufs = list(model.buffers())
        self.saved = [b.clone() for b in self.bufs]

    def restore(self):
        self.arena.flat.copy_(self.flat)
        torch._foreach_copy_(self.bufs, self.saved)
        self.arena.refresh_bf16()


def dump_outputs(out_dir, logs):
    """What the last timed train step computed, for comparing two builds output for output on the same seeded inputs
    (the step starts from InitialState): every value train_step returned to its caller, as `<name>.npy` (float64
    scalar). The weights the step leaves behind are not dumped: AdamW moves each of them by about lr with the sign of its
    gradient, so wherever a gradient is within round-off of zero two runs of one build already differ."""
    os.makedirs(out_dir, exist_ok=True)
    for k, v in logs.items():
        np.save(os.path.join(out_dir, k.replace(os.sep, '_') + '.npy'), np.asarray(float(v), dtype=np.float64))


def _trainable(k, v):
    """Parameters the reference trains: everything but running stats, the frozen 2D stem/stage 1 and the 2D BNs."""
    if not v.is_floating_point() or 'running_' in k or 'num_batches' in k:
        return False
    if k.startswith('backbone.'):
        tail = k[len('backbone.'):]
        is_conv = tail.endswith('.weight') and ('.conv' in tail or '.downsample.0' in tail) and tail.startswith('layer')
        return is_conv and not tail.startswith('layer1.')      # stem (conv1/bn1) + stage 1 frozen, BNs in eval
    return True


def oracle_step(sd, cfg, scan, backward=True):
    """One CPU step of the oracle port on one scan: forward + loss (+ backward through autograd)."""
    from oracle import model_ref as M
    imgs = M.preprocess_imgs(scan['img'][None].cpu(), cfg['data_preprocessor']['mean'], cfg['data_preprocessor']['std'])
    if backward:
        for k, v in sd.items():
            v.requires_grad_(_trainable(k, v))
    losses = M.detector_loss(sd, cfg, [scan['points'].cpu()], imgs, [scan['data_sample']])
    total = sum(losses.values())
    if backward:
        total.backward()
        for v in sd.values():
            v.grad = None
    return float(total.detach())


def cpu_baseline(cfg, variant_args, budget_s=30.0, backward=True, max_steps=None, warmup=0):
    """Oracle port timed on the host cores on a bounded sample (whole scans of the same shape). The warm-up steps double
    as the thread-count calibration: one scan at min(32, nproc) threads and one at all host threads, the faster count runs
    the timed steps and both timings are reported (torch-CPU thrashes on the path's many tiny ops at 128 threads)."""
    from embodiedscan_b200 import MODELS
    from embodiedscan_b200.synth import synth_scan
    torch.manual_seed(0)
    nproc = os.cpu_count() or 1
    sd = {k: v.detach().clone().float() for k, v in MODELS.build(cfg).state_dict().items()}
    scan = synth_scan(0, device='cpu', **variant_args)
    tried = {}
    cores = min(nproc, 32)
    if warmup >= 2:        # two warm-up scans = the thread-count calibration (the in-bench cpu_baseline leg passes 1: no calibration)
        for c in sorted({min(nproc, 32), nproc}):
            torch.set_num_threads(c)
            t0 = time.perf_counter()
            oracle_step(sd, cfg, scan, backward)
            tried[c] = time.perf_counter() - t0
        cores = min(tried, key=tried.get)
        for _ in range(max(0, min(warmup - len(tried), 1))):      # at most one more untimed scan: each costs ~10 s
            oracle_step(sd, cfg, scan, backward)
    torch.set_num_threads(cores)
    n, t0 = 0, time.perf_counter()
    while True:
        oracle_step(sd, cfg, scan, backward)
        n += 1
        el = time.perf_counter() - t0
        if el > budget_s or (max_steps is not None and n >= max_steps) or el / n * (n + 1) > 1.15 * budget_s:
            break
    return {'value': n / el, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'host_threads': nproc,
            'seconds_per_scan_by_threads': {str(k): round(v, 2) for k, v in tried.items()},
            'sample': f'{n} scan(s) of the workload shape, forward + loss' + (' + backward' if backward else '') +
                      ' (no optimiser step), oracle restatement in torch-CPU fp32 — the reference stack '
                      '(MinkowskiEngine / mmcv / pytorch3d / mmdet / mmengine) is not installable here',
            'seconds': el, 'steps_run': n}


def cpu_baseline_subprocess(args, timeout_s=200):
    """Run the CPU port in a child process so a slow host cannot stall the GPU measurement."""
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', '2', '--warmup', '1',
           '--views', str(args.views), '--height', str(args.height), '--width', str(args.width), '--points',
           str(args.points), '--variant', args.variant]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='', RANK='0', WORLD_SIZE='1')
    try:
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, env=env)
        line = [l for l in p.stdout.splitlines() if l.startswith('{')][-1]
        return json.loads(line)['cpu_baseline']
    except Exception as e:  # noqa
        return {'value': None, 'unit': UNIT, 'cores': min(os.cpu_count() or 1, 32), 'kind': 'port',
                'sample': f'unavailable: {type(e).__name__} within {timeout_s}s'}


def run_reference(args):
    """The reference arm: the CPU port of the path on the host cores; one step = one scan of the workload shape (forward +
    loss + backward). The run is bounded to ~150 s of timed work: `steps` in the printed line is what was actually timed."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    from embodiedscan_b200.synth import mv_det3d_config
    v = VARIANTS[args.variant]
    if v['kind'] != 'det':
        print(json.dumps({'impl': 'reference', 'metric': v['metric'], 'unavailable':
                          f'the CPU port is timed for the mv-3ddet workloads (C2, C5); {args.variant} has parity oracles only'}))
        return
    cfg = mv_det3d_config('C2')
    va = dict(n_views=args.views, H=args.height, W=args.width, n_points=args.points)
    base = cpu_baseline(cfg, va, budget_s=150.0, backward=True, max_steps=args.steps, warmup=args.warmup)
    out = {'metric': v['metric'], 'value': base['value'], 'unit': UNIT, 'n_gpus': args.gpus, 'steps': base['steps_run'],
           'steps_requested': args.steps, 'warmup': args.warmup, 'ms_per_step': 1000.0 / base['value'],
           'higher_is_better': True, 'scaling': 'weak',
           'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'impl': 'reference',
           'config': {'workload': f'{args.variant}: mv-3ddet 1 scan/step x {args.views} views {args.height}x{args.width}, '
                                  f'{args.points} points, CPU port'},
           'cpu_baseline': base,
           'e2e': {'value': base['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
           'gpu_launches': 0}
    print(json.dumps(out))


def main():
    args = parse()
    if args.impl == 'reference':
        return run_reference(args)
    if args.row_order:
        os.environ['ESB200_ROW_ORDER'] = args.row_order

    import torch.distributed as dist
    from embodiedscan_b200 import MODELS, _ffi
    from embodiedscan_b200 import sparse as SP
    from embodiedscan_b200.engine import OptimWrapper, broadcast_parameters
    from embodiedscan_b200.synth import mv_det3d_config, synth_scan

    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    dtype = torch.bfloat16 if args.dtype == 'bf16' else torch.float32
    sampler = ClockSampler(local)    # NVML attaches here, long before the timed region (attaching stalls launches briefly)
    sampler.sample()
    sampler.sm.clear()
    torch.manual_seed(0)
    V = VARIANTS[args.variant]
    kind = V['kind']
    va = dict(n_views=args.views, H=args.height, W=args.width, n_points=args.points)
    if kind == 'det':
        cfg = mv_det3d_config('C2')
        opt = dict(lr=1e-3, weight_decay=1e-4, max_norm=10.0)
    elif kind == 'occ':
        from embodiedscan_b200.synth import mv_occ_config, synth_occupancy
        cfg = mv_occ_config('C3')
        opt = dict(lr=1e-4, weight_decay=1e-2, max_norm=35.0)
    else:
        from embodiedscan_b200.synth import add_grounding_prompt, mv_grounding_config
        os.environ.setdefault('ESB200_TEXT_RANDOM_INIT', '1')     # synthetic benchmark: shapes, not RoBERTa's checkpoint
        cfg = mv_grounding_config('C4')
        opt = dict(lr=5e-4, weight_decay=5e-4, max_norm=10.0)
    model = MODELS.build(dict(cfg, compute_dtype=dtype)).to(dev).train()
    optim = OptimWrapper(model, max_run_ahead=args.run_ahead, **opt)
    broadcast_parameters(optim.arena)
    initial = InitialState(model, optim.arena) if args.dump_outputs else None

    n_distinct = 2
    batches = []
    for j in range(n_distinct):
        scans = [synth_scan(1000 * rank + args.batch * j + i, augment=(kind != 'occ'), device=dev, **va)
                 for i in range(args.batch)]
        for i, sc in enumerate(scans):
            if kind == 'occ':
                sc['data_sample'].gt_occupancy = synth_occupancy(sc['data_sample'], cfg['point_cloud_range'],
                                                                 cfg['n_voxels']).to(dev)
            elif kind == 'ground':
                add_grounding_prompt(sc['data_sample'], 1 + (args.batch * j + i) % 3, seed=args.batch * j + i)
        batches.append(scans)

    def device_batch(j):
        scans = batches[j % n_distinct]
        return dict(inputs=dict(points=[s['points'] for s in scans], img=[s['img'] for s in scans]),
                    data_samples=[s['data_sample'] for s in scans])

    def step(j):
        return model.train_step(device_batch(j), optim)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    log(f'model + {n_distinct} batches ready')
    if args.torch_profile:
        from torch.profiler import ProfilerActivity, profile
        for j in range(3):
            step(j)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA], with_stack=True) as prof:
            for j in range(2):
                step(j)
            torch.cuda.synchronize()
        with open(args.torch_profile + (f'.rank{rank}' if world > 1 else ''), 'w') as f:
            f.write(prof.key_averages().table(sort_by='cuda_time_total', row_limit=60, max_name_column_width=70))
            f.write('\n\n')
            f.write(prof.key_averages().table(sort_by='self_cpu_time_total', row_limit=40, max_name_column_width=70))
            f.write('\n\n# by call site (innermost 3 Python frames), sorted by device time, then by host time\n')
            f.write(prof.key_averages(group_by_stack_n=3).table(sort_by='cuda_time_total', row_limit=70,
                                                                max_name_column_width=50, max_src_column_width=110))
            f.write('\n\n')
            f.write(prof.key_averages(group_by_stack_n=3).table(sort_by='self_cpu_time_total', row_limit=70,
                                                                max_name_column_width=50, max_src_column_width=110))
        log('torch profile written')
    for j in range(n_distinct):      # setup pass: one step per distinct batch shape (allocator / cuDNN plan caches)
        step(j)
    for j in range(args.warmup):
        step(j)
        log(f'warmup step {j} done')
    # roofline pass: the same K steps with a CUDA-event pair around every sparse-conv launch (on the launching
    # stream), run BEFORE the timed region and kept out of `value` because ~1.7k event pairs per step cost host time in a host-bound step.
    SP.CONV_PROFILE['records'].clear()
    SP.CONV_PROFILE['enabled'] = True
    model.overlap_2d_3d = False      # time the sparse-conv kernels alone on the device, not sharing SMs with the 2D stream
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    for j in range(args.steps):
        step(args.warmup + j)
    r1.record()
    barrier()
    SP.CONV_PROFILE['enabled'] = False
    model.overlap_2d_3d = True
    ms_roof = r0.elapsed_time(r1)
    log('roofline pass done')
    barrier()
    # clocks are sampled (NVML, main thread) twice during the pre-roll — the same workload under the same load — and ONCE in
    # the middle of the timed region: every NVML query was followed by a 60-140 ms stall of the next step
    sample_at = {} if os.environ.get('ESB_BENCH_NOSAMPLE') == '1' else {max(args.steps // 2, 0)}
    prof_range = os.environ.get('ESB_CUDA_PROFILER_RANGE') == '1'    # for `ncu --profile-from-start off`
    if prof_range:
        torch.cuda.profiler.start()
    import gc
    gc.collect()
    gc.freeze()        # setup objects (model, batches, profile records) leave the collector's working set
    # pre-roll: after an idle period (barrier, gc, event bookkeeping of the roofline pass) single steps stall for 40-400 ms
    # during roughly the next half second (seen at N = 1 and N = 2 alike, never later): run through it before timing
    n_pre = max(3, min(args.steps, 20))
    pre_t = [time.perf_counter()]
    for j in range(n_pre):
        step(j)
        if j in (n_pre // 3, 2 * n_pre // 3):
            sampler.sample()
        pre_t.append(time.perf_counter())
    torch.cuda.synchronize()
    log('host ms per pre-roll step: ' + ' '.join(f'{1e3 * (b - a):.1f}' for a, b in zip(pre_t[:-1], pre_t[1:])))
    if os.environ.get('ESB_BENCH_AUTOGC') == '1':     # A/B: the interpreter's automatic collector instead of the engine's schedule
        gc.enable()
    gc0 = [g['collections'] for g in gc.get_stats()]
    _ffi.launch_counter.update(kernels=0, calls=0, by_name={})
    host_t = [time.perf_counter()]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for j in range(args.steps):
        if initial is not None and j == args.steps - 1:
            initial.restore()
        logs = step(args.warmup + j)
        if j in sample_at:
            ts = time.perf_counter()
            sampler.sample()          # under load, inside the timed region
            log(f'clock sample at timed step {j}: {1e3 * (time.perf_counter() - ts):.2f} ms')
        host_t.append(time.perf_counter())
    e1.record()
    barrier()
    log('gc collections during the timed region (gen0, gen1, gen2): ' +
        ' '.join(str(b['collections'] - a) for a, b in zip(gc0, gc.get_stats())))
    log('host ms per timed step: ' + ' '.join(f'{1e3 * (b - a):.1f}' for a, b in zip(host_t[:-1], host_t[1:])))
    if prof_range:
        torch.cuda.profiler.stop()
    log('timed region done')
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, logs)
        log(f'outputs of timed step {args.steps - 1} written to {args.dump_outputs}')
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms)
    launches = _ffi.launch_counter['kernels']
    value = world * args.batch * args.steps / (ms_total / 1000.0)


    # roofline of the sparse-conv kernels from the events recorded above. Pair model (SURVEY §8d, the contract number):
    # P*(Cin+Cout)*e + 8P + K*Cin*Cout*e per launch; compulsory lower bound (every row read / written once):
    # N_in*Cin*e + N_out*Cout*e + K*Cin*Cout*e (the wgrad output is fp32: K*Cin*Cout*4).
    e = 2 if dtype == torch.bfloat16 else 4
    tot_bytes = tot_ms = tot_flops = tot_comp = 0.0
    n_rec = 0
    wg_bytes = wg_ms = wg_comp = 0.0
    pair_cache = {}
    for kind_, koff, K_, cin, cout, _dt, a, b, n_in, n_out in SP.CONV_PROFILE['records']:
        if id(koff) not in pair_cache:
            pair_cache[id(koff)] = int(koff[-1].item())
        P = pair_cache[id(koff)]
        by = P * (cin + cout) * e + 8 * P + K_ * cin * cout * e
        t = a.elapsed_time(b)
        if kind_ == 'wgrad':
            wg_bytes += by
            wg_ms += t
            wg_comp += n_in * cin * e + n_out * cout * e + K_ * cin * cout * 4
        else:
            # dgrad records carry (cin, cout) already swapped: rows read = the map's output side
            rows_r, rows_w = (n_in, n_out) if kind_ == 'fwd' else (n_out, n_in)
            tot_comp += rows_r * cin * e + rows_w * cout * e + K_ * cin * cout * e
            tot_bytes += by
            tot_ms += t
            tot_flops += 2.0 * P * cin * cout
            n_rec += 1
    peak, peak_src = peaks()
    achieved = tot_bytes / (tot_ms / 1000.0) / 1e9 if tot_ms > 0 else 0.0
    agg = (tot_bytes + wg_bytes) / ((tot_ms + wg_ms) / 1000.0) / 1e9 if tot_ms + wg_ms > 0 else 0.0
    traffic, traffic_note = None, None
    for name in ('r2_traffic.json', 'r1_traffic.json'):
        tpath = os.path.join(ROOT, 'profiles', name)
        if os.path.exists(tpath):
            tj = json.load(open(tpath)).get('spconv_tc_fwd_kernel')
            if tj:
                traffic, traffic_note = tj['dram_bytes_per_launch_avg'], tj['source']
                break
    roofline = {'bound': 'hbm', 'kernel': 'spconv_tc_fwd_kernel (tcgen05; forward + dgrad launches)', 'achieved': achieved,
                'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic, 'traffic_note': traffic_note,
                'algorithmic_bytes_per_launch_avg': tot_bytes / max(n_rec, 1), 'peak_source': peak_src,
                'launches_timed': n_rec, 'avg_launch_us': 1000.0 * tot_ms / max(n_rec, 1),
                'achieved_tflops': tot_flops / (tot_ms / 1000.0) / 1e12 if tot_ms > 0 else 0.0,
                'share_of_step': tot_ms / ms_roof, 'pass_ms_per_step': ms_roof / args.steps,
                'wgrad_achieved_gbs': wg_bytes / (wg_ms / 1000.0) / 1e9 if wg_ms > 0 else 0.0,
                'wgrad_frac': (wg_bytes / (wg_ms / 1000.0) / 1e9 / peak) if wg_ms > 0 else 0.0,
                'wgrad_share_of_step': wg_ms / ms_roof,
                'aggregate_achieved_gbs': agg, 'aggregate_frac': agg / peak,
                'aggregate_note': 'forward + dgrad + wgrad launches together (what SURVEY §8d states the 60% target on)',
                'compulsory_bytes_per_launch_avg': tot_comp / max(n_rec, 1),
                'compulsory_frac': (tot_comp / (tot_ms / 1000.0) / 1e9 / peak) if tot_ms > 0 else 0.0,
                'compulsory_note': 'same launches and times, bytes = every input / output row and the filter moved once '
                                   '(N_in*Cin*e + N_out*Cout*e + K*Cin*Cout*e): the gather re-reads of the pair model are '
                                   'served by the 126 MB L2, so this is the fraction of HBM peak the kernel needs',
                'measured': 'separate pass over the same K steps with per-launch CUDA events, 2D/3D stream overlap off so each '
                            'kernel is timed alone on the device (excluded from value)'}

    # end to end: pinned host inputs -> H2D -> train_step -> loss read back, every step
    e2e = None
    if not args.no_e2e:
        host = []
        for scans in batches:
            host.append(dict(points=[s['points'].cpu().pin_memory() for s in scans],
                             img=[s['img'].cpu().pin_memory() for s in scans]))
        h2d = sum(t.numel() * t.element_size() for t in host[0]['points'] + host[0]['img'])

        def e2e_step(j):
            hb = host[j % n_distinct]
            data = dict(inputs=dict(points=hb['points'], img=hb['img']),
                        data_samples=[s['data_sample'] for s in batches[j % n_distinct]])
            lg = model.train_step(data, optim)
            return float(lg['loss'])       # device -> host read of the step's result

        log('e2e warmup')
        for j in range(max(args.warmup, 3)):
            e2e_step(j)
        barrier()
        log('e2e timed')
        t0 = time.perf_counter()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for j in range(args.steps):
            e2e_step(j)
        g1.record()
        barrier()
        wall = torch.tensor([max(time.perf_counter() - t0, g0.elapsed_time(g1) / 1000.0)], device=dev)
        if world > 1:
            dist.all_reduce(wall, op=dist.ReduceOp.MAX)
        e2e = {'value': world * args.batch * args.steps / float(wall), 'unit': UNIT, 'h2d_bytes_per_step': h2d,
               'd2h_bytes_per_step': 4}

    out = {'metric': V['metric'], 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
           'ms_per_step': ms_total / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
           'dtype': args.dtype, 'data': 'synthetic',
           'config': {'workload': f'{args.variant}: train step, {args.batch} scans/GPU x {args.views} views '
                                  f'{args.height}x{args.width} RGB-D, {args.points} points/scan, {V["model"]}, AdamW + clip',
                      'global_batch': world * args.batch, 'parallelism': f'dp{world}',
                      'row_order': os.environ.get('ESB200_ROW_ORDER', 'input'), 'run_ahead': args.run_ahead,
                      'l2': 'per-step working set (340 MB fp32 weights + multi-GB activations) exceeds the 126 MB L2; '
                            f'{n_distinct} distinct input batches alternate; {n_distinct} untimed setup steps precede the W warm-up steps',
                      'loss': {k: float(v) for k, v in logs.items()}},
           'clocks': sampler.summary(), 'gpu_launches': launches, 'roofline': roofline, 'impl': 'esb200'}
    if e2e is not None:
        out['e2e'] = e2e
    if rank == 0 and world == 1 and not args.no_cpu_baseline and kind == 'det':
        log('cpu baseline (oracle port, subprocess with a hard timeout)')
        out['cpu_baseline'] = cpu_baseline_subprocess(args, timeout_s=200)
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
