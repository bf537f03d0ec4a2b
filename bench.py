#!/usr/bin/env python
"""bench.py — VirConv-L backbone scenes/s (forward+backward) on synthetic KITTI-shaped scenes.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" = one forward+backward pass of the VirConv-L 3-D backbone (20 sparse convs + BN/ReLU + 4x index2uv,
scalar loss = sum of mean features of x_conv1..4 and the encoded tensor) over one batch of 2 synthetic
scenes per GPU (BASELINE.json configs[1]: 16k LiDAR + 80k virtual points per scene, 40 000-voxel cap,
reference grid [81,1600,1408]).  One JSON line on rank 0 (contract: task statement "Measurement").

  value     scenes/s with inputs resident in HBM, per-step CUDA-event time, max over ranks
  e2e       same step driven from PINNED HOST buffers: H2D of voxel features/coords/params, D2H of the loss
  roofline  the dominant kernel (gather-GEMM: conv forward + dgrad launches): algorithmic bytes / event time
  cpu_baseline / --impl reference : the restated reference algorithm (spconv "Native": CPU hash-map rulebook +
            per-offset torch.mm + index_add_) from oracle/, timed on this box's host cores.

--dump-outputs DIR writes what the last timed step of `value` computed, as a caller of the step receives it: the loss
(DIR/loss.npy) and every parameter gradient (DIR/grad.<parameter name>.npy), float32.  Inputs and initial weights are
seeded, so two builds run with the same arguments can be compared output for output.  The gradients are accumulated
with float atomics, so two runs of one build already differ slightly (bf16, on a B200 at 1000 W: loss bit-identical,
gradients up to 3.4e-3 of a tensor's largest element apart).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CFG = dict(RETURN_NUM_FEATURES_AS_DICT=True, OUT_FEATURES=64, LAYER_DISCARD_RATE=0.1, NUM_FILTERS=[16, 32, 64, 64])
SCENES_PER_GPU = 2          # VirConv-L.yaml:284 BATCH_SIZE_PER_GPU
N_LIDAR, N_VIRTUAL, MAX_VOXELS = 16384, 80000, 40000
POOL = 4                    # distinct batches rotated through the timed steps
WORKLOAD = ('VirConv-L 3D backbone fwd+bwd, synthetic KITTI scenes 16k LiDAR + 80k virtual pts, '
            '40000-voxel cap/scene, grid [81,1600,1408], batch 2/GPU')


class _StdoutToStderr:
    """OS-level redirect of fd 1 to fd 2 while NCCL initialises: with NCCL_DEBUG=VERSION|WARN in the environment the library
    prints its version banner on stdout, where the driver expects exactly one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)
        return False



def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20, help='timed steps per measurement (at least 1)')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--precision', default=os.environ.get('VIRCONV_PRECISION', 'bf16'), choices=['fp32', 'bf16'],
                    help='bf16 = tcgen05 tensor-core contractions (BASELINE configs[1] dtype); fp32 = 1e-4 parity kernels')
    ap.add_argument('--ref-budget-s', type=float, default=150.0)
    ap.add_argument('--cpu-worker', action='store_true', help=argparse.SUPPRESS)
    ap.add_argument('--cpu-thread-sweep', action='store_true', help='CPU arm at several thread counts (profiles/ evidence)')
    ap.add_argument('--model', default='L', choices=['L', 'T'],
                    help='L = VirConv-L (VirConvL8x; the headline metric, BASELINE configs[1]); T = VirConv-T / -S backbone '
                         '(VirConv8x, MM stream + LiDAR stream: BASELINE configs[2] and [4]) — training step and ROT_NUM=3 eval '
                         'forward, gradient all-reduce timed separately (exposed time)')
    ap.add_argument('--mode', default=os.environ.get('VIRCONV_BENCH_MODE', 'graph'), choices=['graph', 'eager'],
                    help='graph = the whole step (forward + loss + backward) replayed as one CUDA graph (plan executor static '
                         'mode: device row counts, no host synchronisation); eager = exact-shape execution, one C-ABI call per '
                         'forward / backward, 4 data-dependent row counts read on the host')
    ap.add_argument('--tc-variant', type=int, default=int(os.environ.get('VIRCONV_TC_VARIANT', '1')), choices=[0, 1],
                    help='A/B aid: 1 = persistent tensor-core kernels (default), 0 = the round-1 kernels')
    ap.add_argument('--wgrad-variant', type=int, default=int(os.environ.get('VIRCONV_WGRAD_VARIANT', '1')), choices=[0, 1],
                    help='A/B aid: 1 = wgrad_tc3.cu (half-tile stages, shares SMs with the dgrad kernels; default), 0 = wgrad_tc2.cu')
    ap.add_argument('--wgrad-ctas', type=int, default=0)
    ap.add_argument('--bn-fused', type=int, default=1, choices=[0, 1], help='A/B aid: BatchNorm backward as one cooperative launch (1) or two (0)')
    ap.add_argument('--no-grid41', action='store_true', help='skip the extra [41,1600,1408]-grid measurement (N=1, graph mode)')
    ap.add_argument('--graph-pipeline', type=int, default=int(os.environ.get('VIRCONV_GRAPH_PIPELINE', '0')), choices=[0, 1],
                    help='graph mode: 1 = graph.PipelinedStep (index graph of step t+1 beside the feature graph of step t), 0 = one graph per step')
    ap.add_argument('--ncu-step', action='store_true',
                    help='profiling aid: W warm-up steps, then exactly one step between cudaProfilerStart/Stop; no JSON')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='VirConv-L: write the loss and parameter gradients of the last timed step as DIR/<name>.npy')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and (a.impl != 'ours' or a.model != 'L' or a.ncu_step):
        ap.error('--dump-outputs applies to the VirConv-L measurement of --impl ours')
    return a


def dump_outputs(out_dir, loss, named_params):
    """The step's outputs as float32 .npy files: loss.npy and grad.<parameter name>.npy (zeros for a parameter the loss
    does not reach)."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'loss.npy'), loss.detach().float().reshape(1).cpu().numpy())
    for name, p in named_params:
        g = p.grad if p.grad is not None else torch.zeros_like(p)
        np.save(os.path.join(out_dir, f'grad.{name}.npy'), g.detach().float().cpu().numpy())


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
             'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix='.csv')
        self.proc = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(gpu_index), f'--query-gpu={self.QUERY}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(',')]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle's CPU restatement (the only place bench.py executes oracle/)
# ------------------------------------------------------------------------------------------------------
def cpu_step(model, batch):
    vf = torch.from_numpy(batch.voxel_features.copy())
    vc = torch.from_numpy(batch.voxel_coords.copy())
    model.zero_grad(set_to_none=True)
    o = model(vf, vc, batch.batch_size, batch.calib, batch.aug_param)
    loss = o['out'].features.mean() + sum(o['x_conv%d' % i].features.mean() for i in range(1, 5))
    loss.backward()
    return float(loss.detach())


def cpu_threads():
    """Threads for the CPU legs: the per-offset mm / index_add_ of the Native algorithm stop scaling (and then slow
    down) beyond a few tens of threads, so 'all the threads it can use' is the count that is FASTEST on the B200 box's
    128-core host: 16 (sweep, profiles/cpu_thread_sweep_r2.txt from `python bench.py --cpu-thread-sweep`: 0.98 scenes/s at
    4 threads, 1.28 at 8, 1.50 at 16, 1.05 at 32, 0.39 at 64, 0.01 at 128).  VIRCONV_CPU_THREADS overrides."""
    env = os.environ.get('VIRCONV_CPU_THREADS')
    if env:
        return max(1, int(env))
    return max(1, min(os.cpu_count() or 1, 16))


def run_cpu_thread_sweep():
    """scenes/s of the CPU arm for a range of thread counts (one warm-up + 3 steps each)."""
    from virconv_b200 import scenes
    cm = make_cpu_model()
    b = scenes.make_batch([0, 1], N_LIDAR, N_VIRTUAL, MAX_VOXELS, training=True)
    n = os.cpu_count() or 1
    for t in [c for c in (4, 8, 16, 32, 64) if c <= n]:          # (128 threads: 200 s per step on the B200 box's host)
        torch.set_num_threads(t)
        cpu_step(cm, b)
        ts = []
        for _ in range(3):
            t0 = time.time()
            cpu_step(cm, b)
            ts.append(time.time() - t0)
        print(f'threads {t:4d}: {SCENES_PER_GPU / float(np.mean(ts)):.3f} scenes/s ({1e3 * float(np.mean(ts)):.0f} ms/step)', flush=True)


def run_cpu_worker():
    from virconv_b200 import scenes
    cores = cpu_threads()
    torch.set_num_threads(cores)
    cm = make_cpu_model()
    b = scenes.make_batch([0, 1], N_LIDAR, N_VIRTUAL, MAX_VOXELS, training=True)
    cpu_step(cm, b)                                   # warm-up (thread pools, allocator)
    budget, times = 20.0, []
    t0 = time.time()
    while not times or (time.time() - t0 + times[-1] < budget and len(times) < 12):
        t = time.time()
        cpu_step(cm, b)
        times.append(time.time() - t)
    dt = float(np.mean(times))
    print(json.dumps({'value': SCENES_PER_GPU / dt, 'unit': 'scenes/s', 'cores': cores, 'kind': 'port',
                      'sample': f'{len(times)} fwd+bwd steps of one batch of {SCENES_PER_GPU} scenes of the same workload '
                                f'({sum(times):.1f} s, mean {dt:.2f} s/step, after 1 warm-up step), restated reference '
                                f'algorithm (oracle/), {cores} threads of {os.cpu_count()} host cores'}), flush=True)


def make_cpu_model():
    from oracle import spconv_cpu
    from oracle.backbone import VirConvL8x as OracleL
    spconv_cpu.RULEBOOK_BACKEND = 'c'            # sequential hash-map indexing, like spconv's CPU path
    torch.manual_seed(666)
    m = OracleL()
    m.train()
    return m


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from virconv_b200 import scenes
    cores = cpu_threads()
    torch.set_num_threads(cores)
    model = make_cpu_model()
    batches = [scenes.make_batch([2 * i, 2 * i + 1], N_LIDAR, N_VIRTUAL, MAX_VOXELS, training=True) for i in range(2)]
    t0 = time.time()
    n_warm = 0
    for w in range(max(args.warmup, 1)):
        cpu_step(model, batches[w % 2])
        n_warm += 1
        if time.time() - t0 > 0.4 * args.ref_budget_s:        # (a very slow host: keep most of the budget for timed steps)
            break
    warm = time.time() - t0
    per = max(warm / n_warm, 1e-3)
    k = max(1, min(args.steps, int(max(args.ref_budget_s - warm, per) / per)))
    times = []
    for s in range(k):
        t = time.time()
        cpu_step(model, batches[s % 2])
        times.append(time.time() - t)
    ms = 1e3 * float(np.mean(times))
    val = SCENES_PER_GPU / (ms / 1e3)
    sample = (f'{k} step(s) of one batch of {SCENES_PER_GPU} scenes (same workload), after {n_warm} warm-up step(s); '
              f'steps capped by a {args.ref_budget_s:.0f} s budget')
    line = {'impl': 'reference', 'metric': 'VirConv-L scenes/sec (fwd+bwd)', 'value': val, 'unit': 'scenes/s',
            'n_gpus': args.gpus, 'steps': k, 'warmup': n_warm, 'ms_per_step': ms, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'scenes_per_step': SCENES_PER_GPU,
                       'what': 'restated reference algorithm on CPU (spconv Native: C hash-map rulebook + per-offset '
                               'torch.mm + index_add_, autograd backward); spconv itself is not installable here'},
            'cpu_baseline': {'value': val, 'unit': 'scenes/s', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': val, 'unit': 'scenes/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# VirConv-T / VirConv-S backbone (BASELINE configs[2], [4]): separate arm, not the headline metric
# ------------------------------------------------------------------------------------------------------
CFG_T = dict(RETURN_NUM_FEATURES_AS_DICT=True, OUT_FEATURES=64, LAYER_DISCARD_RATE=0.15, NUM_FILTERS=[16, 32, 64, 64], MM=True)
MAX_VOXELS_T_TRAIN, MAX_VOXELS_T_TEST = 16000, 40000      # VirConv-T.yaml:120-121


def run_ours_t(args):
    """VirConv8x (`spconv_backbone.py:232-535`): training step (one pass per stream, batch 2/GPU, random init — config 5
    "VirConv-S training step": the two models share this backbone) with the gradient all-reduce timed on its own, and the
    ROT_NUM=3 eval forward (LiDAR stream x-batched, MM stream looped — config 3).  Exact-shape executor path (one C-ABI call
    per plan forward / backward); the CUDA-graph static mode covers VirConv-L only so far."""
    import torch.distributed as dist
    from virconv_b200 import _lib, ops, parallel, scenes
    from virconv_b200.backbone import VirConv8x
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        with _StdoutToStderr():
            dist.init_process_group('nccl', device_id=dev)
            dist.barrier()
    lib = _lib.load()
    torch.manual_seed(666)
    model = VirConv8x(CFG_T, 8, [1408, 1600, 80], precision=args.precision).to(dev).train()
    params = list(model.parameters())
    if world > 1:
        for p in params:
            dist.broadcast(p.data, 0)

    def to_dev(b, train):
        bd = {k: torch.from_numpy(v).to(dev) for k, v in b.arrays.items()}
        bd.update(batch_size=b.batch_size, calib=b.calib)
        if train:
            bd['aug_param'] = torch.from_numpy(b.aug_param)
        else:
            bd['transform_param'] = torch.from_numpy(b.transform_param)
        return bd

    train_b = [to_dev(scenes.make_batch_mm(parallel.shard_scene_ids(i, rank, world, SCENES_PER_GPU), N_LIDAR, N_VIRTUAL,
                                           MAX_VOXELS_T_TRAIN, training=True), True) for i in range(POOL)]
    test_b = [to_dev(scenes.make_batch_mm(parallel.shard_scene_ids(100 + i, rank, world, SCENES_PER_GPU), N_LIDAR, N_VIRTUAL,
                                          MAX_VOXELS_T_TEST, training=False, rot_num=3), False) for i in range(2)]
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def loss_of(out, sfx=('',)):
        loss = 0
        for s_ in sfx:
            loss = loss + out['encoded_spconv_tensor' + s_].features.mean()
            for grp in ('multi_scale_3d_features', 'multi_scale_3d_features_mm'):
                for t in out[grp + s_].values():
                    if t is not None:
                        loss = loss + t.features.mean()
        return loss

    def train_step(bd, reduce=True):
        for p in params:
            p.grad = None
        out = model(dict(bd))
        loss = loss_of(out)
        loss.backward()
        ar = None
        if reduce and world > 1:
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            parallel.allreduce_gradients(params, average=True)
            e.record()
            ar = (a, e)
        return loss, ar

    def timed_train(n, reduce=True):
        evs, ars = [], []
        for s_ in range(n):
            flush_buf.zero_()
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            _, ar = train_step(train_b[s_ % POOL], reduce)
            e.record()
            evs.append((a, e))
            if ar:
                ars.append(ar)
        torch.cuda.synchronize()
        return [a.elapsed_time(e) for a, e in evs], [a.elapsed_time(e) for a, e in ars]

    def timed_eval(n):
        model.eval()
        evs = []
        with torch.no_grad():
            for s_ in range(n):
                flush_buf.zero_()
                a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                model(dict(test_b[s_ % 2]))
                e.record()
                evs.append((a, e))
        torch.cuda.synchronize()
        model.train()
        return [a.elapsed_time(e) for a, e in evs]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    timed_train(max(args.warmup, 3))
    barrier()
    timed_train(args.steps)                  # allocator priming
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = lib.vc_launch_count()
    ms_list, ar_list = timed_train(args.steps)
    launches = (lib.vc_launch_count() - l0) / max(args.steps, 1)
    barrier()
    ms_nored, _ = timed_train(args.steps, reduce=False)
    barrier()
    timed_eval(3)
    ev_list = timed_eval(max(args.steps // 2, 4))
    barrier()
    clocks = sampler.stop() if sampler else None
    tot = torch.tensor([sum(ms_list) / len(ms_list), sum(ms_nored) / len(ms_nored), sum(ev_list) / len(ev_list),
                        (sum(ar_list) / len(ar_list)) if ar_list else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    err = int(ops.tc_error_flag(dev).item())
    assert err == 0, 'tensor-core pipeline timeout flag set'
    if rank == 0:
        ms_step, ms_step_nored, ms_eval, ms_ar = [float(x) for x in tot]
        n_par = sum(p.numel() for p in params)
        line = {'metric': 'VirConv-T/S backbone scenes/sec (fwd+bwd)', 'value': SCENES_PER_GPU * world / (ms_step * 1e-3),
                'unit': 'scenes/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms_step,
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'bf16' if args.precision == 'bf16' else 'f32', 'data': 'synthetic', 'gpu_launches': launches,
                'config': {'workload': 'VirConv-T / VirConv-S 3D backbone (VirConv8x: LiDAR stream + MM stream) fwd+bwd, synthetic KITTI '
                                       'scenes 16k LiDAR + 80k virtual pts, 16000-voxel cap per stream and scene (train), grid '
                                       '[81,1600,1408], batch 2/GPU, random init',
                           'scenes_per_step': SCENES_PER_GPU * world, 'parallelism': f'dp{world}',
                           'l2': 'flushed between timed steps (256 MiB write)', 'timing': 'per-step CUDA events, max over ranks'},
                'allreduce': {'bytes': 4 * n_par, 'ms': ms_ar, 'exposed_ms': max(ms_step - ms_step_nored, 0.0),
                              'ms_per_step_without_allreduce': ms_step_nored,
                              'note': 'one flat fp32 bucket (NCCL AVG) after the backward: nothing overlaps it, exposed = its own time'},
                'eval_rot3': {'ms_per_forward': ms_eval, 'scenes_per_s': SCENES_PER_GPU * world / (ms_eval * 1e-3),
                              'what': 'ROT_NUM=3 test-mode forward: LiDAR stream x-batched [D,H,4W], MM stream 3 passes, 40000-voxel cap'},
                'clocks': clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def run_ours(args):
    if args.model == 'T':
        return run_ours_t(args)
    import torch.distributed as dist
    from virconv_b200 import _lib, ops, parallel, scenes
    from virconv_b200.backbone import VirConvL8x

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (the product has no CPU path); use --impl reference for the CPU arm')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        with _StdoutToStderr():
            dist.init_process_group('nccl', device_id=dev)
            dist.barrier()                      # (communicator creation — and NCCL's banner — happen here)
    lib = _lib.load()
    _lib.check(lib.vc_set_tc_variant(int(args.tc_variant)), 'vc_set_tc_variant')
    _lib.check(lib.vc_conv_wgrad_tc3_config(int(args.wgrad_variant), int(args.wgrad_ctas)), 'vc_conv_wgrad_tc3_config')
    _lib.check(lib.vc_set_bn_fused(int(args.bn_fused)), 'vc_set_bn_fused')

    torch.manual_seed(666)
    model = VirConvL8x(CFG, 8, [1408, 1600, 80], precision=args.precision).to(dev).train()
    params = [p for p in model.parameters()]
    if world > 1:
        for p in params:
            dist.broadcast(p.data, 0)

    host, devb = [], []
    h2d = 0
    for i in range(POOL):
        b = scenes.make_batch(parallel.shard_scene_ids(i, rank, world, SCENES_PER_GPU), N_LIDAR, N_VIRTUAL, MAX_VOXELS,
                              training=True)
        hv = torch.from_numpy(b.voxel_features).pin_memory()
        hc = torch.from_numpy(b.voxel_coords).pin_memory()
        host.append((hv, hc, b))
        devb.append((hv.to(dev), hc.to(dev), b))
        h2d = hv.numel() * 4 + hc.numel() * 4 + b.batch_size * 28 * 4
    # graph mode: the step starts one stage earlier, at the collated raw points (`batch_dict['points']`, dataset.py:349-353):
    # hash-grid voxelisation + MeanVFE (vc_voxelize_mean, the GPU replacement of the dataloader's Point2VoxelCPU3d) run inside
    # the captured step, so the e2e H2D payload is the point cloud itself
    VOX = dict(point_cloud_range=(0, -40, -3, 70.4, 40, 1), voxel_size=(0.05, 0.05, 0.05), max_points_per_voxel=5,
               max_voxels=MAX_VOXELS, vfe_model='max')
    host_p, dev_p = [], []
    if args.mode == 'graph':
        for i in range(POOL):
            pb = scenes.make_points_batch(parallel.shard_scene_ids(i, rank, world, SCENES_PER_GPU), N_LIDAR, N_VIRTUAL, training=True)
            hp = torch.from_numpy(pb.points).pin_memory()
            host_p.append((hp, pb))
            dev_p.append((hp.to(dev), pb))
            h2d = hp.numel() * 4 + pb.batch_size * 28 * 4
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    from virconv_b200.graph import GraphedStep, masked_mean

    def loss_of(out):
        loss = masked_mean(out['encoded_spconv_tensor'])
        for t in out['multi_scale_3d_features'].values():
            loss = loss + masked_mean(t)
        return loss

    ar_events = []

    def reduce_grads():
        """one flat fp32 bucket over NCCL / NVLink (no-op at N=1); runs on the main stream right after the backward, so its
        whole duration is exposed — measured with events and reported as config.allreduce_ms_per_step"""
        if world == 1:
            return
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        parallel.allreduce_gradients(params, average=True)
        e.record()
        ar_events.append((a, e))

    def step(vf, vc, b, sync_loss, resident=False):
        """exact-shape (eager) step: one C-ABI call per forward / backward"""
        for p in params:
            p.grad = None
        bd = {'voxel_features': vf, 'voxel_coords': vc, 'batch_size': b.batch_size, 'calib': b.calib,
              'aug_param': b.aug_param,
              # resident int32 coordinates (the `value` loop): this step's rulebook pipeline may overlap the previous
              # step's backward; the e2e loop uploads on the main stream every step and makes no such promise
              'virconv_inputs_ready': resident}
        out = model(bd)
        loss = loss_of(out)
        loss.backward()
        reduce_grads()
        return float(loss.detach()) if sync_loss else loss

    # capacity head-room of the captured step's buffers over the first batch's row counts: every kernel of the static mode works on
    # (or zero-fills) capacity-sized buffers, so head-room costs time (1.3: 2.98 ms/step, 1.05: 2.91); a batch that does not fit
    # re-captures with more (all POOL batches pass through the untimed warm-up steps first)
    MARGIN = float(os.environ.get('VIRCONV_GRAPH_MARGIN', '1.15'))
    if args.mode == 'graph' and args.graph_pipeline:
        from virconv_b200.graph import PipelinedStep
        graphed = PipelinedStep(model, loss_of, params, margin=MARGIN, voxelizer=VOX)
    else:
        graphed = GraphedStep(model, loss_of, params, margin=MARGIN, voxelizer=VOX) if args.mode == 'graph' else None

    def gstep(pts, pb):
        """graph step: the collated points (device or pinned-host tensor) are copied into the graph's input buffer, then ONE
        graph launch: voxelise + VFE -> rulebooks -> 20 x (conv, BN, ReLU) -> loss -> backward"""
        loss = graphed({'points': pts, 'batch_size': pb.batch_size, 'calib': pb.calib, 'aug_param': pb.aug_param})
        reduce_grads()
        return loss

    # e2e upload targets: a ring of device buffers (what a prefetching loader keeps), so the timed loop allocates nothing
    # (a cudaMalloc landing inside it costs 30-60 ms: profiles/e2e_repeat_r1.txt).  Slot reuse is safe: the executor never
    # lets the host run more than 4 forwards ahead of the GPU.  (graph mode copies straight into the graph's input buffers)
    RING = 8
    n_max = max(h[0].shape[0] for h in host)
    ring = [(torch.empty((n_max, host[0][0].shape[1]), dtype=torch.float32, device=dev),
             torch.empty((n_max, host[0][1].shape[1]), dtype=host[0][1].dtype, device=dev)) for _ in range(RING)]
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream(dev)
    loss_host = torch.zeros(4096, dtype=torch.float32).pin_memory()
    last_loss = [None]

    def timed(n_steps, from_host):
        """from_host (the e2e loop): every step uploads its inputs from PINNED host memory and reads its loss back into
        pinned host memory, both inside the timed region — the way a training loop with a prefetching loader and lagged
        loss logging does it; nothing blocks the host per step, all copies have completed when the timed region ends
        (synchronize below).  eager mode: the upload runs on a copy stream (the main and rulebook streams wait for its
        event); graph mode: the upload goes straight into the graph's input buffers on the main stream."""
        evs = []
        for s in range(n_steps):
            flush_buf.zero_()
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            if from_host:
                hv, hc, b = host[s % POOL]
                if graphed is not None:
                    loss = gstep(*host_p[s % POOL])
                else:
                    rf, rc = ring[s % RING]
                    vf, vc = rf[:hv.shape[0]], rc[:hc.shape[0]]
                    with torch.cuda.stream(copy_stream):
                        vf.copy_(hv, non_blocking=True)
                        vc.copy_(hc, non_blocking=True)
                        up = torch.cuda.Event()
                        up.record(copy_stream)
                    main_stream.wait_event(up)
                    ops.side(dev).stream.wait_event(up)        # the executor's rulebook stream reads the coordinates
                    loss = step(vf, vc, b, False, resident=True)
                loss_host[s % loss_host.numel()].copy_(loss.detach(), non_blocking=True)
            else:
                vf, vc, b = devb[s % POOL]
                if graphed is not None:
                    loss = gstep(*dev_p[s % POOL])
                else:
                    loss = step(vf, vc, b, False, resident=True)
            last_loss[0] = loss
            e.record()
            evs.append((a, e))
        torch.cuda.synchronize()
        if from_host:
            assert bool(torch.isfinite(loss_host[:min(n_steps, loss_host.numel())]).all()), 'non-finite loss read back'
        err = int(ops.tc_error_flag(dev).item())
        assert err == 0, 'a tensor-core pipeline wait timed out (error flag %d): results are invalid' % err
        return [a.elapsed_time(e) for a, e in evs]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.ncu_step:
        timed(max(args.warmup, 1), False)
        torch.cuda.profiler.start()
        timed(1, False)
        torch.cuda.profiler.stop()
        return
    timed(max(args.warmup, 3), False)
    barrier()
    # allocator priming (untimed, after the W warm-up steps): the timed loop below never synchronises, so the host runs
    # several steps ahead of the GPU and that many per-step arenas are in flight at once; let the caching allocator create
    # those blocks now rather than with cudaMalloc calls inside the timed region (seen as 5-10 ms/step outliers)
    sampler = ClockSampler(local) if rank == 0 else None      # samples the priming burst too (same load, more samples)
    timed(args.steps, False)
    barrier()
    dev_allocs0 = torch.cuda.memory_stats(dev).get('num_device_alloc', 0)
    l0 = lib.vc_launch_count()
    t_wall = time.time()
    del ar_events[:]
    ms_list = timed(args.steps, False)
    barrier()
    wall = time.time() - t_wall
    ar_ms = sum(a.elapsed_time(e) for a, e in ar_events) / max(len(ar_events), 1) if ar_events else 0.0
    launches = (lib.vc_launch_count() - l0) / max(args.steps, 1)
    if graphed is not None:
        launches = graphed.launches_per_replay        # kernels of this library inside the captured step (counted at capture)
    dev_allocs = torch.cuda.memory_stats(dev).get('num_device_alloc', 0) - dev_allocs0
    if args.dump_outputs and rank == 0:
        # before anything else runs a step: the graph's loss and the .grad tensors are rewritten by every step
        dump_outputs(args.dump_outputs, last_loss[0], model.named_parameters())
    timed(max(2, min(args.steps, 10)), True)      # warm-up + allocator priming of the e2e loop
    barrier()
    st0 = torch.cuda.memory_stats(dev)
    e2e_list = timed(args.steps, True)
    barrier()
    st1 = torch.cuda.memory_stats(dev)
    e2e_allocs = {k: int(st1.get(k, 0) - st0.get(k, 0)) for k in ('num_device_alloc', 'num_device_free', 'num_alloc_retries',
                                                                   'num_sync_all_streams')}
    clocks = sampler.stop() if sampler else None

    tot = torch.tensor([sum(ms_list), sum(e2e_list)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    ms_step = float(tot[0]) / args.steps
    ms_e2e = float(tot[1]) / args.steps
    scenes_per_step = SCENES_PER_GPU * world

    # roofline pass: the same step with CUDA events around every conv kernel launch (not part of the timed loops).
    # Plan-executor path: the events are recorded inside vc_exec_forward / vc_exec_backward (executor.timing_*);
    # module path (VIRCONV_EXECUTOR=0): around every conv C-ABI call (ops.KernelTimer).
    from virconv_b200 import executor
    roof, kern, run = None, {}, None
    nprof = 3
    use_exec = executor.ENABLED
    if rank == 0 and not use_exec:
        ops.TIMER = ops.KernelTimer()
    # kernels are timed ALONE here: one stream, no concurrent wgrad (in the timed loops above the executor overlaps the
    # index / feature / wgrad streams, which stretches every individual kernel and is not what a roofline describes)
    saved = (executor.TWO_STREAMS, executor.WGRAD_STREAM)
    executor.TWO_STREAMS, executor.WGRAD_STREAM = False, False
    for s in range(nprof):               # every rank runs the steps (they contain the gradient all-reduce)
        flush_buf.zero_()
        vf, vc, b = devb[s % POOL]
        if rank == 0 and use_exec:
            executor.timing_start()
        step(vf, vc, b, False)
        if rank == 0 and use_exec:
            run = executor.LAST_RUN
            for kind, layer, ms in executor.timing_stop():
                by, fl = executor.alg_bytes_flops(run, kind, layer)
                c = kern.setdefault(kind, [0, 0.0, 0, 0])
                c[0] += 1
                c[1] += ms
                c[2] += by
                c[3] += fl
            executor.LAST_RUN = None
    executor.TWO_STREAMS, executor.WGRAD_STREAM = saved
    barrier()
    if rank == 0 and use_exec and run is not None:
        sys.stderr.write('plan executor arena: %.0f MB used of %.0f MB per step\n' % (run.query(0, 0)[0] / 2**20, run.arena.numel() / 2**20))
    if rank == 0:
        if not use_exec:
            kern = ops.TIMER.summary()
            ops.TIMER = None
        peak, how = peaks()
        dom = ('conv_fwd_tc', 'conv_dgrad_tc') if args.precision == 'bf16' else ('conv_fwd', 'conv_dgrad')
        g_calls = sum(kern[k][0] for k in dom if k in kern)
        g_ms = sum(kern[k][1] for k in dom if k in kern)
        g_bytes = sum(kern[k][2] for k in dom if k in kern)
        g_flops = sum(kern[k][3] for k in dom if k in kern)
        all_ms = sum(v[1] for v in kern.values())
        ach = g_bytes / (g_ms * 1e-3) / 1e9 if g_ms > 0 else 0.0
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, 'profiles', 'traffic_tc_gather.json' if args.precision == 'bf16' else 'traffic_gather_f32.json')
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get('dram_bytes_per_launch')     # from the committed ncu --set full capture
            traffic_src = 'profiles/' + os.path.basename(tp) + ' (ncu --set full capture of this kernel, not measured in this run)'
        roof = {'bound': 'hbm', 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak, 'traffic': traffic,
                'traffic_source': traffic_src,
                'kernel': ('tc_conv_persist_kernel<KC,NR> (persistent tcgen05 conv forward + gather dgrad)'
                           if args.precision == 'bf16' else
                           'gather_gemm_kernel<CI,CO> (fp32 conv forward + dgrad), prep_weights included'),
                'peak_source': how, 'launches_per_step': g_calls / nprof,
                'avg_launch_ms': g_ms / max(g_calls, 1), 'alg_bytes_per_launch': g_bytes / max(g_calls, 1),
                'achieved_tflops': g_flops / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0,
                'share_of_conv_kernel_time': g_ms / all_ms if all_ms > 0 else None,
                'per_step_ms': {k: v[1] / nprof for k, v in kern.items()},
                'note': ('tcgen05 bf16 operands / fp32 TMEM accumulators; bytes = bf16 gathered operand + fp32 output + P*8 '
                         '+ bf16 weights; CUDA events around each launch inside the plan executor, kernels timed alone (single stream)'
                         if args.precision == 'bf16' else
                         'fp32 CUDA-core parity path: FP32-FMA bound, HBM is the bound it is designed toward')}

    roof_w = None
    if rank == 0 and roof is not None and kern.get('conv_wgrad_tc'):
        c, ms, by, fl = kern['conv_wgrad_tc']
        peak, how = peaks()
        roof_w = {'bound': 'hbm', 'kernel': ('tc_wgrad_half_kernel<CI,CO> (persistent tcgen05 weight gradient, half-tile stages, 74 CTAs: sized to '
                                            'run beside the main stream, timed alone here)' if args.wgrad_variant == 1 else
                                            'tc_wgrad_persist_kernel<CI,CO> (persistent tcgen05 weight gradient, one CTA per SM)'),
                  'achieved': by / (ms * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s', 'frac': by / (ms * 1e-3) / 1e9 / peak,
                  'launches_per_step': c / nprof, 'avg_launch_ms': ms / max(c, 1), 'alg_bytes_per_launch': by / max(c, 1),
                  'achieved_tflops': fl / (ms * 1e-3) / 1e12, 'peak_source': how,
                  'note': 'bytes = bf16 gathered rows + bf16 dout + P*8 + fp32 gradient; CUDA events inside the plan executor, kernels alone'}

    # the same workload on BASELINE's wording of the grid, [41,1600,1408] (0.1 m z voxels; SURVEY §8d config 2 asks for both):
    # its own model instance (sparse_shape is a model attribute) and captured step, N=1 only, same timing rules
    grid41 = None
    if world == 1 and graphed is not None and not args.no_grid41:
        torch.manual_seed(666)
        model41 = VirConvL8x(CFG, 8, [1408, 1600, 40], precision=args.precision).to(dev).train()
        vs41 = (0.05, 0.05, 0.1)
        vox41 = dict(VOX, voxel_size=vs41)
        g41 = GraphedStep(model41, loss_of, list(model41.parameters()), margin=MARGIN, voxelizer=vox41)
        pts41 = []
        for i in range(POOL):
            pb = scenes.make_points_batch(parallel.shard_scene_ids(i, rank, world, SCENES_PER_GPU), N_LIDAR, N_VIRTUAL, training=True,
                                          voxel_size=vs41)
            pts41.append((torch.from_numpy(pb.points).to(dev), pb))

        def run41(n):
            evs = []
            for s_ in range(n):
                flush_buf.zero_()
                a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                pts, pb = pts41[s_ % POOL]
                g41({'points': pts, 'batch_size': pb.batch_size, 'calib': pb.calib, 'aug_param': pb.aug_param})
                e.record()
                evs.append((a, e))
            torch.cuda.synchronize()
            return sum(a.elapsed_time(e) for a, e in evs) / n
        run41(max(args.warmup, 3))
        ms41 = run41(args.steps)
        grid41 = {'value': scenes_per_step / (ms41 * 1e-3), 'unit': 'scenes/s', 'ms_per_step': ms41,
                  'workload': WORKLOAD.replace('[81,1600,1408]', '[41,1600,1408]') + ' (z voxel 0.1 m)', 'captures': g41.recaptures}
        del g41, model41, pts41

    # the same captured step WITHOUT the voxeliser inside (device-resident voxel features / coordinates, what round 1's `value`
    # timed and what the reference's dataloader hands the model): N=1 only, same timing rules
    from_voxels = None
    if world == 1 and graphed is not None and not args.no_grid41:
        gv = GraphedStep(model, loss_of, params, margin=MARGIN)

        def runv(n):
            evs = []
            for s_ in range(n):
                flush_buf.zero_()
                a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                vf, vc, b = devb[s_ % POOL]
                gv({'voxel_features': vf, 'voxel_coords': vc, 'batch_size': b.batch_size, 'calib': b.calib, 'aug_param': b.aug_param})
                e.record()
                evs.append((a, e))
            torch.cuda.synchronize()
            return sum(a.elapsed_time(e) for a, e in evs) / n
        runv(max(args.warmup, 3))
        msv = runv(args.steps)
        from_voxels = {'value': scenes_per_step / (msv * 1e-3), 'unit': 'scenes/s', 'ms_per_step': msv, 'captures': gv.recaptures,
                       'what': 'the graph-replayed step starting from pre-voxelised device-resident inputs (no voxeliser inside)'}
        del gv

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cpu_base = None
    if world == 1 and not args.no_cpu_baseline:
        # bounded sample in a child process (so a slow host cannot take the bench line down with it)
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), '--cpu-worker'], capture_output=True, text=True,
                               timeout=240)
            cpu_base = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as ex:          # noqa: BLE001
            cpu_base = {'value': None, 'unit': 'scenes/s', 'cores': cpu_threads(), 'kind': 'port',
                        'sample': f'CPU baseline did not finish inside its 240 s bound ({type(ex).__name__})'}

    line = {'metric': 'VirConv-L scenes/sec (fwd+bwd)', 'value': scenes_per_step / (ms_step * 1e-3), 'unit': 'scenes/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms_step,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16' if args.precision == 'bf16' else 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'scenes_per_step': scenes_per_step, 'parallelism': f'dp{world}',
                       'allreduce_ms_per_step': ar_ms,       # gradient all-reduce (exposed: main stream, after the backward)
                       'host_path': ('whole step (forward + loss + backward) replayed as ONE CUDA graph: plan executor static mode, '
                                     'device row counts, no host synchronisation; %d capture(s)' % graphed.recaptures
                                     if graphed is not None else
                                     'native plan executor: one C-ABI call per forward / backward, index ops on a side stream'
                                     if executor.ENABLED else 'per-operator C-ABI calls from Python autograd'),
                       'l2': 'flushed between timed steps (256 MiB write)', 'timing': 'per-step CUDA events, max over ranks',
                       'e2e_loop': ('graph mode: the collated raw points (pinned host memory) are uploaded into the graph\'s input buffer '
                                    'every step, voxelisation + VFE run inside the graph, the loss is copied back to pinned host '
                                    'memory every step (asynchronous, completed inside the timed region)' if graphed is not None else
                                    'inputs uploaded from pinned host memory on a copy stream every step, loss copied back to '
                                    'pinned host memory every step (asynchronous, completed inside the timed region)'),
                       'step_input': ('raw points [N, 1+8] -> vc_voxelize_mean inside the step' if graphed is not None else
                                      'host-pre-voxelised features + coordinates'),
                       'precision': ('bf16 operands on tcgen05 for conv forward/dgrad (C>=16), fp32 accumulate, fp32 features, '
                                     'fp32 wgrad/BN' if args.precision == 'bf16' else 'fp32 storage, fp32 accumulate (parity path)')},
            'e2e': {'value': scenes_per_step / (ms_e2e * 1e-3), 'unit': 'scenes/s', 'ms_per_step': ms_e2e,
                    'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': 4 + 4 * 4, 'allocator_events_in_timed_region': e2e_allocs},
            'gpu_launches': launches, 'wall_s_timed_region': wall,
            'value_wall_clock': scenes_per_step * args.steps / wall,      # includes the L2 flushes and inter-step gaps
            'cuda_mallocs_in_timed_region': int(dev_allocs), 'clocks': clocks, 'roofline': roof,
            'roofline_wgrad': roof_w, 'value_grid41': grid41, 'value_from_voxels': from_voxels, 'cpu_baseline': cpu_base}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    a = parse()
    if a.cpu_worker:
        run_cpu_worker()
    elif a.cpu_thread_sweep:
        run_cpu_thread_sweep()
    elif a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
