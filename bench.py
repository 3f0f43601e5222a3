#!/usr/bin/env python
"""Replay-step throughput bench (BASELINE.json metric: replay-step images/sec, ASER+SCR,
Reduced-ResNet18, CIFAR-100 shapes, mem_size 5000).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One *step* = one ER+ASER replay step (BASELINE config 3: asvm, k=3, n_smp_cls 1.5, 10 stream + 10
replayed images) AND one SCR replay step (BASELINE config 2: SupCon temp 0.07, mlp head, 10 stream +
100 replayed images), each on its own learner with its own pre-filled 5000-slot memory; 20 stream
images per step.  Inputs are synthetic (uniform images, uniform labels), weights random-init.

  value  stream images/sec with the stream batches already resident in HBM
  e2e    the same through the public plugin API with HOST batches: pinned host -> device copy of
         every batch and a device -> host read of both losses inside the timed region
  N > 1  data-parallel stream shards: every rank runs its own stream shard and memory, gradients are
         averaged with one NCCL all-reduce of the flat gradient arena per optimizer step (weak scaling)
  --impl reference   the reference's algorithm on the host CPU cores (oracle/replay_step.py, the
         restatement pinned against the reference's agents) when oracle/_ref is absent
  --dump-outputs DIR   after the timed steps, write what the last device-resident step left a caller
         (both losses, weights, BN statistics, memory labels, a seeded sample of memory images) as
         DIR/<name>.npy, so that two builds can be compared output for output on identical inputs
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True           # the tree may be read-only: nothing is written into it

WORKLOAD = ('ER+ASER replay step (asvm,k=3,n_smp_cls=1.5,10+10 imgs) + SCR replay step '
            '(SupCon T=0.07,mlp head,10+100 imgs x 2 views), CIFAR-100 shapes, mem_size 5000, batch 10')
MEM_SIZE = 5000
BATCH = 10
NUM_CLASSES = 100
TRICK = {'labels_trick': False, 'kd_trick': False, 'separated_softmax': False, 'review_trick': False,
         'ncm_trick': False, 'kd_trick_star': False}


def params_for(kind):
    base = dict(data='cifar100', cuda=True, epoch=1, batch=BATCH, verbose=False, mem_size=MEM_SIZE, mem_iters=1,
                k=3, aser_type='asvm', n_smp_cls=1.5, num_tasks=10, buffer_tracker=False, optimizer='SGD',
                learning_rate=0.1, weight_decay=0, temp=0.07, head='mlp', subsample=50, error_analysis=False,
                trick=dict(TRICK))
    if kind == 'aser':
        base.update(agent='ER', retrieve='ASER', update='ASER', eps_mem_batch=10)
    else:
        base.update(agent='SCR', retrieve='random', update='random', eps_mem_batch=100)
    return SimpleNamespace(**base)


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {'hbm_gbs': p['hbm_gbs'], 'bf16_tflops': p['bf16_tflops'],
                'bf16_tflops_sustained': p.get('bf16_tflops_sustained', p['bf16_tflops']), 'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.FIELDS,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


# ----------------------------------------------------------------------------- CUDA arm
def build_learner(kind, seed):
    import torch
    from b200ocl import nets, registry
    from b200ocl.memory import ClassBalancedRandomSampling as CB
    p = params_for(kind)
    model = nets.setup_architecture(p)
    learner = registry.agents[p.agent](model, None, p)
    g = torch.Generator(device='cuda').manual_seed(seed)
    buf = learner.buffer
    buf.buffer_img.copy_(torch.rand(buf.buffer_img.shape, device='cuda', generator=g))
    labels = np.random.RandomState(seed).randint(0, NUM_CLASSES, MEM_SIZE).astype(np.int64)
    buf.buffer_label.copy_(torch.from_numpy(labels).cuda())
    buf.labels_host[:] = labels
    buf.current_index = MEM_SIZE
    buf.n_seen_so_far = MEM_SIZE + BATCH            # > mem_size: ASER retrieval is active (aser_retrieve.py:24)
    if kind == 'aser':
        CB.reset()
        CB.update_cache(buf.buffer_label, NUM_CLASSES, new_y=labels, ind=np.arange(MEM_SIZE))
    learner.model.train()
    return learner


def run_ours(args, rank, world):
    import torch
    import torch.distributed as dist
    from b200ocl import _native, ops
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    np.random.seed(1000 + rank)
    torch.manual_seed(1000 + rank)
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):       # stdout carries exactly one JSON line
        aser = build_learner('aser', 10 + rank)
        scr = build_learner('scr', 20 + rank)
    if world > 1:
        # same initial weights on every rank, then gradient averaging keeps the replicas identical
        for L in (aser, scr):
            dist.broadcast(L.engine.state.params, src=0)
            dist.broadcast(L.engine.state.bn_stats, src=0)
            L.engine.pack()
            L.grad_sync = lambda eng: dist.all_reduce(eng.state.grads)
            L.grad_world = world
    total = args.warmup + args.steps
    rs = np.random.RandomState(7 + rank)
    host_x = torch.from_numpy(rs.rand(2 * total, BATCH, 3, 32, 32).astype(np.float32)).pin_memory()
    host_y = rs.randint(0, NUM_CLASSES, (2 * total, BATCH)).astype(np.int64)
    host_y_pin = torch.from_numpy(host_y).pin_memory()
    dev_x = host_x.to(dev)
    dev_y = torch.from_numpy(host_y).to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2

    mids = []

    def step(i, from_host):
        if from_host:
            xa = host_x[2 * i].to(dev, non_blocking=True); xs = host_x[2 * i + 1].to(dev, non_blocking=True)
            ya = host_y_pin[2 * i].to(dev, non_blocking=True); ys = host_y_pin[2 * i + 1].to(dev, non_blocking=True)
        else:
            xa, xs, ya, ys = dev_x[2 * i], dev_x[2 * i + 1], dev_y[2 * i], dev_y[2 * i + 1]
        aser.replay_step(xa, ya, host_y[2 * i])
        if mids is not None and len(mids) < 4096:
            m = torch.cuda.Event(enable_timing=True)
            m.record()
            mids.append(m)
        scr.replay_step(xs, ys, host_y[2 * i + 1])
        if from_host:
            return float(aser.last_loss), float(scr.last_loss)       # device -> host read of the step's result
        return None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(from_host):
        for i in range(args.warmup):
            step(i, from_host)
        from b200ocl import engine as _eng
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()                           # BEFORE the barrier: spawning nvidia-smi must not delay rank 0's step 0
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        barrier()
        launches0 = _native.launch_count() + _eng.graph_launch_count()
        t0 = time.perf_counter()
        del mids[:]
        for k in range(args.steps):
            flush.fill_(k & 255)                      # L2 flush between timed iterations (outside the event pair)
            ev[k][0].record()
            step(args.warmup + k, from_host)
            ev[k][1].record()
        barrier()
        split = {'aser_ms': float(np.median([a.elapsed_time(m) for (a, _), m in zip(ev, mids)])),
                 'scr_ms': float(np.median([m.elapsed_time(b) for (_, b), m in zip(ev, mids)]))}
        wall = time.perf_counter() - t0
        clocks = sampler.stop() if rank == 0 else None
        per_step = torch.tensor([a.elapsed_time(b) for a, b in ev], dtype=torch.float64, device=dev)
        t = torch.cat([per_step.sum().reshape(1), per_step])
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)          # MAX over ranks of the sum and of every step
        steps_ms = np.sort(t[1:].cpu().numpy())
        stats = {'median_ms': float(np.median(steps_ms)), 'p10_ms': float(steps_ms[int(0.1 * (len(steps_ms) - 1))]),
                 'p90_ms': float(steps_ms[int(round(0.9 * (len(steps_ms) - 1)))]), 'max_ms': float(steps_ms[-1])}
        stats.update(split)
        return float(t[0].item()), _native.launch_count() + _eng.graph_launch_count() - launches0, clocks, wall, stats

    log('rank %d: learners built' % rank)
    ms_dev, launches, clocks, wall, stats = timed(False)
    log('rank %d: device-resident pass %.2f ms/step' % (rank, ms_dev / args.steps))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'aser': aser, 'scr': scr})
    ms_e2e, _, _, _, stats_e2e = timed(True)
    log('rank %d: end-to-end pass %.2f ms/step' % (rank, ms_e2e / args.steps))
    if rank != 0:
        return None
    imgs = 2 * BATCH * world * args.steps
    # per-kernel-class device time of one step (separate pass, event-bracketed inside the library)
    from b200ocl import engine as _engine
    _graphs_were = _engine._GRAPHS
    _engine.set_graphs(False)                 # the per-launch profiler needs eager launches (same kernels)
    from b200ocl import learners as _learners
    _conc_were = _learners._CONCURRENT
    _learners.set_concurrent(False)           # ... on one stream: a class time must not contain another stream's kernels
    prof = profile_step(lambda i: step(i, False), args.warmup + args.steps - 1) if world == 1 else None
    _learners.set_concurrent(_conc_were)
    _engine.set_graphs(_graphs_were)
    pk = peaks()
    line = {
        'metric': 'replay-step images/sec (ASER+SCR, ResNet18, CIFAR100)', 'value': imgs / (ms_dev * 1e-3),
        'unit': 'stream images/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD,
                   'stream_images_per_step': 2 * BATCH, 'trained_images_per_step': 20 + 110,
                   'parallelism': 'dp%d stream shards, NCCL grad all-reduce' % world if world > 1 else 'single GPU',
                   'l2': 'flushed (256 MiB write) between timed steps', 'wall_s_timed_region': wall,
                   'step_ms': stats, 'e2e_step_ms': stats_e2e},
        'e2e': {'value': imgs / (ms_e2e * 1e-3), 'unit': 'stream images/s',
                'h2d_bytes_per_step': 2 * (BATCH * 3 * 32 * 32 * 4 + BATCH * 8), 'd2h_bytes_per_step': 8},
        'gpu_launches': int(launches), 'clocks': clocks,
    }
    if prof is not None:
        line['roofline'] = prof['roofline']
        line['kernel_ms_per_step'] = prof['classes']
    return line


def dump_outputs(out_dir, learners, n_img_rows=256):
    """What the last timed step left a caller of replay_step: its loss, the weights and BatchNorm running
    statistics of the model, the memory's labels and a fixed, seeded sample of the memory's image rows
    (the whole memory is 61 MB per learner).  float32 arrays as computed; labels and losses as float64."""
    import torch
    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    for name, L in learners.items():
        buf = L.buffer
        rows = np.sort(np.random.RandomState(0).choice(buf.buffer_img.shape[0], n_img_rows, replace=False))
        arrays = {'loss': np.array([float(L.last_loss)], dtype=np.float64),
                  'params': L.engine.state.params.cpu().numpy(),
                  'bn_stats': L.engine.state.bn_stats.cpu().numpy(),
                  'buffer_label': buf.buffer_label.cpu().numpy().astype(np.float64),
                  'buffer_img_rows': rows.astype(np.float64),
                  'buffer_img_sample': buf.buffer_img[torch.from_numpy(rows).to(buf.buffer_img.device)].cpu().numpy()}
        for k, a in arrays.items():
            np.save(os.path.join(out_dir, '%s_%s.npy' % (name, k)), a)
    log('outputs of the last timed step written to %s' % out_dir)


def profile_step(step_fn, i):
    """Device time per kernel class for one step, CUDA events recorded around every launch by the
    library on its launch stream (b200ocl_profile_*).  Returns the roofline object for the class with
    the largest share."""
    import torch
    from b200ocl import _native
    lib = _native.lib()
    if not hasattr(lib, 'b200ocl_profile_begin'):
        return None
    torch.cuda.synchronize()
    lib.b200ocl_profile_begin()
    step_fn(i)
    torch.cuda.synchronize()
    import ctypes
    n = lib.b200ocl_profile_end()
    classes = {}
    name = ctypes.create_string_buffer(64)
    ms, cnt, work = ctypes.c_double(), ctypes.c_int(), ctypes.c_double()
    for k in range(n):
        lib.b200ocl_profile_get(k, name, 64, ctypes.byref(ms), ctypes.byref(cnt), ctypes.byref(work))
        classes[name.value.decode()] = {'ms': ms.value, 'launches': cnt.value, 'work': work.value}
    if not classes:
        return None
    top = max(classes, key=lambda c: classes[c]['ms'])
    pk = peaks()
    c = classes[top]
    total_ms = sum(v['ms'] for v in classes.values())
    if top.startswith('conv') or top.startswith('wgrad'):
        achieved = c['work'] / (c['ms'] * 1e-3) / 1e12 if c['ms'] > 0 else 0.0      # work = FLOPs
        roof = {'kernel': top, 'bound': 'tensor', 'achieved': achieved, 'peak': pk['bf16_tflops_sustained'],
                'unit': 'TFLOP/s', 'frac': achieved / pk['bf16_tflops_sustained'], 'traffic': None,
                'peak_source': pk['source'] + ' cuBLAS bf16 (sustained); ' +
                               ('conv_tcp issues 3 TF32 tcgen05 passes per useful FLOP (fp32-grade 3xTF32), so its '
                                'tensor-pipe work is ~3.4x the useful FLOPs counted here' if top == 'conv_tcp'
                                else 'this kernel computes in fp32 on the CUDA cores'),
                'traffic_note': ('dram read+write of one ncu --set full capture of this kernel (N = 210, 20->20 ch, '
                                 '32x32): 17.3 MB per launch for 17.2 MB of input; see profiles/r01_v4_conv_tcp.md'
                                 if top == 'conv_tcp' else None),
                'share_of_step': c['ms'] / total_ms, 'avg_launch_us': 1e3 * c['ms'] / max(c['launches'], 1)}
        if top not in ('conv_tcp', 'conv_tc', 'conv_tc_train'):
            # fp32 CUDA-core kernel: the pipe that bounds it is the FMA pipe, not the tensor pipe
            fp32_peak = 148 * 128 * 2 * 1965.0e6 / 1e12
            roof['fp32_fma'] = {'achieved_tflops': achieved, 'peak_tflops': fp32_peak, 'frac': achieved / fp32_peak,
                                'peak_source': '148 SMs x 128 FMA lanes x 2 x 1965 MHz'}
        if top == 'conv_tcp':
            # issued work: 3 TF32 passes per useful FLOP, by-product halo rows and padded channel slots (x3.4 at these shapes);
            # the TF32 dense peak is half of the measured bf16 figure
            roof['achieved_issued_tf32'] = achieved * 3.4
            roof['frac_issued_vs_tf32_peak'] = achieved * 3.4 / (pk['bf16_tflops_sustained'] / 2.0)
    else:
        achieved = c['work'] / (c['ms'] * 1e-3) / 1e9 if c['ms'] > 0 else 0.0       # work = bytes
        roof = {'kernel': top, 'bound': 'hbm', 'achieved': achieved, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                'frac': achieved / pk['hbm_gbs'], 'traffic': None, 'peak_source': pk['source'],
                'share_of_step': c['ms'] / total_ms, 'avg_launch_us': 1e3 * c['ms'] / max(c['launches'], 1)}
    # roofline.traffic: dram read + write bytes per launch of that class from the committed ncu pass (profiles/r02_traffic.json)
    try:
        with open(os.path.join(ROOT, 'profiles', 'r02_traffic.json')) as fh:
            tr = json.load(fh)
        t = tr['classes'].get(top)
        if t:
            roof['traffic'] = t['dram_read_bytes_per_launch'] + t['dram_write_bytes_per_launch']
            roof['traffic_note'] = ('dram__bytes_read.sum + dram__bytes_write.sum per launch, averaged over %d launches of this '
                                    'class: %s' % (t['launches'], tr['command']))
    except (OSError, ValueError, KeyError):
        pass
    return {'roofline': roof, 'classes': {k: round(v['ms'], 4) for k, v in sorted(classes.items(), key=lambda kv: -kv[1]['ms'])}}



# ----------------------------------------------------------------------------- kNN-SV sweep (BASELINE config 5)
def run_knn_sweep(args, rank, world):
    """`--workload knn_sweep`: 50 000 x 512 buffer features against 1 000 candidates, k = 3.  Eval rows (the
    memory) are sharded across the ranks, the candidate block is replicated, each rank runs the fused kernel
    on its shard and ONE NCCL all-gather moves the [3, C] column partials (sharded.knn_sv_sharded); every rank
    combines them in rank order and ranks the candidates.  Strong scaling: the total work is fixed.
    A step = one full sweep.  Rank 0 also runs the unsharded kernel and reports `ok`."""
    import torch
    import torch.distributed as dist
    from b200ocl import ops, sharded
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    E, C, d, k = 50000, 1000, 512, 3
    g = torch.Generator(device=dev).manual_seed(0)          # same data on every rank
    ef = torch.relu(torch.randn(E, d, device=dev, generator=g))
    cf = torch.relu(torch.randn(C, d, device=dev, generator=g))
    ey = torch.randint(0, 100, (E,), device=dev, generator=g)
    cy = torch.randint(0, 100, (C,), device=dev, generator=g)
    lo, hi = sharded.shard_bounds(E, rank, world)
    ef_l, ey_l = ef[lo:hi].contiguous(), ey[lo:hi].contiguous()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def sweep():
        return sharded.aser_scores_sharded(ef_l, ey_l, E, cf, cy, k, 100)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(args.warmup):
        sweep()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for i in range(args.steps):
        flush.fill_(i & 255)
        ev[i][0].record()
        top, red = sweep()
        ev[i][1].record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    per = torch.tensor([a.elapsed_time(b) for a, b in ev], dtype=torch.float64, device=dev)
    t = torch.cat([per.sum().reshape(1), per])
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None
    ms = float(t[0]) / args.steps
    full = ops.knn_sv(ef, ey, cf, cy, k, want_sum=True, want_max=True, want_min=True)
    err = float((full['sum'] - red['sum']).abs().max())
    ok = err < 2e-4 and torch.equal(full['max'], red['max']) and torch.equal(full['min'], red['min'])
    same = float((ops.rank_desc(full['sum'], 100) == top).float().mean())
    pk = peaks()
    alg_bytes = 4.0 * d * (E + C) + 8.0 * (E + C) + 4.0 * C * 3            # SURVEY 8(d): features + labels + 3 reductions
    flops = 3.0 * E * C * d                                                 # direct-difference distances (sub, fma)
    fp32_peak = 148 * 128 * 2 * (clocks['sm_max_mhz'] or 1965.0) * 1e6 / 1e12 if clocks else 74.4
    steps_ms = np.sort(t[1:].cpu().numpy())
    return {
        'metric': 'kNN-SV sweep eval rows/sec (50k x 512 buffer features, 1k candidates, k=3)', 'value': E / (ms * 1e-3),
        'unit': 'eval rows/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'ASER kNN-SV sweep: 50000 x 512 relu(N(0,1)) buffer features, 1000 candidates, labels U{0..99}, '
                               'k=3, column sum/max/min + top-100; eval rows sharded over %d GPU(s), one NCCL all-gather of '
                               '[3,1000] partials' % world,
                   'l2': 'flushed (256 MiB write) between timed steps', 'step_ms': {'median': float(np.median(steps_ms)),
                                                                                    'max': float(steps_ms[-1])}},
        'ok': bool(ok), 'max_abs_err_vs_unsharded': err, 'top100_identical_fraction': same,
        'roofline': {'kernel': 'knn_sv', 'bound': 'hbm', 'achieved': alg_bytes / (ms * 1e-3) / 1e9 / world,
                     'peak': pk['hbm_gbs'], 'unit': 'GB/s', 'frac': alg_bytes / (ms * 1e-3) / 1e9 / world / pk['hbm_gbs'],
                     'traffic': None, 'peak_source': pk['source'],
                     'note': 'per-GPU algorithmic bytes / sweep time.  At d=512 the kernel is compute-bound (arithmetic '
                             'intensity ~490 FLOP/B, SURVEY 7.3-1): see fp32_fma',
                     'fp32_fma': {'achieved_tflops': flops / (ms * 1e-3) / 1e12 / world, 'peak_tflops': fp32_peak,
                                  'frac': flops / (ms * 1e-3) / 1e12 / world / fp32_peak,
                                  'peak_source': '148 SMs x 128 FMA lanes x 2 x max SM clock'}},
        'gpu_launches': 2 * args.steps, 'clocks': clocks,
    }

# ----------------------------------------------------------------------------- CPU arm (reference algorithm)
def build_oracle_state(kind, seed):
    import torch
    from oracle import replay_step as ors
    from oracle import resnet as oresnet
    spec = oresnet.Spec(32, 20, NUM_CLASSES, head='mlp' if kind == 'scr' else None)
    params, bn = oresnet.seeded_state(spec, seed)
    for name in oresnet.bn_names(spec):           # fresh-model statistics
        bn[name + '.running_mean'].zero_(); bn[name + '.running_var'].fill_(1.0)
    st = ors.ReplayState(spec, params, bn, MEM_SIZE, (3, 32, 32), NUM_CLASSES, lr=0.1)
    rs = np.random.RandomState(seed)
    st.buffer_img = torch.from_numpy(rs.rand(MEM_SIZE, 3, 32, 32).astype(np.float32))
    labels = rs.randint(0, NUM_CLASSES, MEM_SIZE).astype(np.int64)
    st.buffer_label = torch.from_numpy(labels)
    st.current_index = MEM_SIZE
    st.n_seen_so_far = MEM_SIZE + BATCH
    if kind == 'aser':
        st.cache_update_bulk = True
        for c in range(NUM_CLASSES):
            st.class_index_cache[c] = set(np.flatnonzero(labels == c).tolist())
            st.class_num_cache[c] = len(st.class_index_cache[c])
    return st


def host_cores():
    """Cores this process may actually use: affinity mask, capped by a cgroup CPU quota if one is set
    (os.cpu_count() reports the machine, which oversubscribes torch's intra-op pool in a container)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        with open('/sys/fs/cgroup/cpu.max') as fh:
            quota, period = fh.read().split()
        if quota != 'max':
            n = max(1, min(n, int(float(quota) / float(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def log(msg):
    print('[bench %7.1fs] %s' % (time.perf_counter() - T0, msg), file=sys.stderr, flush=True)


T0 = time.perf_counter()


def run_reference_harness(device, steps, warmup, timeout_s=600):
    """The UNMODIFIED reference agents (oracle/_ref, compiled by oracle/fetch_ref.py) through
    baseline/ref_harness.py in a subprocess: --device cpu hides the GPUs so that every
    torch.cuda.is_available() gate of the reference is off; --device cuda is the reference's own
    single-GPU PyTorch path (cudnn.deterministic as general_main.py:15-18).  None if the tree is absent."""
    sys.path.insert(0, os.path.join(ROOT, 'baseline'))
    try:
        import ref_harness
    finally:
        sys.path.pop(0)
    if ref_harness.locate() is None:
        return None
    cores = host_cores()
    cmd = [sys.executable, os.path.join(ROOT, 'baseline', 'ref_harness.py'), '--device', device,
           '--steps', str(steps), '--warmup', str(warmup), '--threads', str(cores)]
    env = dict(os.environ)
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_ADDR', 'MASTER_PORT'):
        env.pop(k, None)
    log('reference (%s) arm: %s' % (device, ' '.join(cmd[1:])))
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, env=env)
    except subprocess.TimeoutExpired:
        log('reference (%s) arm timed out' % device)
        return None
    if r.returncode != 0:
        log('reference (%s) arm failed: %s' % (device, r.stderr[-2000:]))
        return None
    out = json.loads(r.stdout.strip().splitlines()[-1])
    log('reference (%s) arm: ASER %.1f ms/step, SCR %.1f ms/step' % (device, out['aser_ms_per_step'], out['scr_ms_per_step']))
    out['cores'] = cores
    return out


def run_reference(args, steps, warmup, budget_s=30.0):
    """The reference's replay step on the host cores.  Preferred: the unmodified reference itself
    (kind "reference"); without oracle/_ref: oracle/replay_step.py, the restatement pinned against it
    (kind "port").  Each step is one ER+ASER step and one SCR step like the CUDA arm."""
    h = run_reference_harness('cpu', steps, warmup)
    if h is not None:
        return {'steps': steps, 'value': h['stream_images_per_s'], 'unit': 'stream images/s', 'cores': h['cores'],
                'kind': 'reference',
                'sample': '%d steps (one ER+ASER + one SCR replay step each) of the same workload after %d warm-up, '
                          '%.1f s of CPU time, unmodified reference agents via train_learner (identity augmentation '
                          'stub: kornia is absent), torch intra-op threads = %d'
                          % (steps, max(warmup, 1), h['seconds'], h['threads']),
                'ms_per_step': h['ms_per_step_pair'], 'aser_ms': h['aser_ms_per_step'], 'scr_ms': h['scr_ms_per_step']}
    return run_reference_port(args, steps, warmup, budget_s)


def run_reference_port(args, steps, warmup, budget_s=30.0):
    import torch
    from oracle import replay_step as ors
    cores = host_cores()
    torch.set_num_threads(cores)
    log('reference arm (port): %d host cores (os.cpu_count()=%s)' % (cores, os.cpu_count()))
    np.random.seed(0); torch.manual_seed(0)
    st_a, st_s = build_oracle_state('aser', 31), build_oracle_state('scr', 32)
    rs = np.random.RandomState(5)

    def step():
        xa = torch.from_numpy(rs.rand(BATCH, 3, 32, 32).astype(np.float32)); ya = torch.from_numpy(rs.randint(0, NUM_CLASSES, BATCH))
        xs = torch.from_numpy(rs.rand(BATCH, 3, 32, 32).astype(np.float32)); ys = torch.from_numpy(rs.randint(0, NUM_CLASSES, BATCH))
        ors.er_step(st_a, xa, ya, retrieve='ASER', update='ASER', eps_mem_batch=10, k=3, aser_type='asvm', n_smp_cls=1)
        ors.scr_step(st_s, xs, ys, eps_mem_batch=100, temperature=0.07)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    done = 0
    while done < steps:
        step()
        done += 1
        if time.perf_counter() - t0 > budget_s:       # bounded sample
            break
    dt = time.perf_counter() - t0
    steps = done
    log('reference arm (port): %d steps in %.1f s' % (steps, dt))
    return {'steps': steps, 'value': 2 * BATCH * steps / dt, 'unit': 'stream images/s', 'cores': cores, 'kind': 'port',
            'sample': '%d steps (one ER+ASER + one SCR replay step each) of the same workload after %d warm-up, '
                      '%.1f s of CPU time, torch intra-op threads = %d' % (steps, warmup, dt, cores),
            'ms_per_step': 1e3 * dt / steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--workload', default='replay', choices=['replay', 'knn_sweep'])
    ap.add_argument('--dump-outputs', metavar='DIR', default=None)
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))

    if args.impl == 'reference':
        if rank != 0:
            return 0
        os.environ['CUDA_VISIBLE_DEVICES'] = ''                      # the CPU arm never touches a GPU
        steps, warmup = args.steps, max(1, args.warmup)
        r = run_reference(args, steps, warmup, budget_s=float('inf'))
        steps = r['steps']
        line = {'impl': 'reference', 'metric': 'replay-step images/sec (ASER+SCR, ResNet18, CIFAR100)',
                'value': r['value'], 'unit': 'stream images/s', 'n_gpus': args.gpus, 'steps': steps, 'warmup': warmup,
                'ms_per_step': r['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f32', 'data': 'synthetic',
                'config': {'workload': WORKLOAD, 'stream_images_per_step': 2 * BATCH, 'trained_images_per_step': 20 + 110,
                           'parallelism': 'host CPU, %d threads' % r['cores']},
                'cpu_baseline': {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
                'e2e': {'value': r['value'], 'unit': 'stream images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'gpu_launches': 0}
        print(json.dumps(line))
        return 0

    # stdout carries exactly ONE JSON line: libraries that write to fd 1 (NCCL prints its version there) go to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + '\n').encode())

    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', int(os.environ.get('LOCAL_RANK', 0))))
    if args.workload == 'knn_sweep':
        line = run_knn_sweep(args, rank, world)
        if rank == 0:
            emit(line)
        if world > 1:
            dist.destroy_process_group()
        return 0
    line = run_ours(args, rank, world)
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            r = run_reference(args, 30, 2, budget_s=20.0)     # ~12 s of CPU work on 16 cores
            line['cpu_baseline'] = {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')}
            g = run_reference_harness('cuda', 40, 5)          # the north-star's >=10x denominator
            if g is not None:
                line['reference_gpu'] = {
                    'value': g['stream_images_per_s'], 'unit': 'stream images/s', 'ms_per_step': g['ms_per_step_pair'],
                    'aser_ms': g['aser_ms_per_step'], 'scr_ms': g['scr_ms_per_step'],
                    'what': 'unmodified reference agents (oracle/_ref) on cuda:0, torch %s eager, '
                            'cudnn.deterministic=True, benchmark=False (general_main.py:15-18), same workload, '
                            '40 steps after 5 warm-up, identity augmentation stub (kornia absent: the reference does '
                            'less work than in production)' % g['torch']}
                line['vs_reference_gpu'] = {'value_ratio': line['value'] / g['stream_images_per_s'],
                                            'e2e_ratio': line['e2e']['value'] / g['stream_images_per_s']}
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
