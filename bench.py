#!/usr/bin/env python
"""Benchmark of the PV-RAFT hot path (BASELINE.json metric: RAFT iters/sec at N=8192, iters=32;
corr-kernel HBM GB/s vs peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]

A "step" is one full `RSF.forward(p, num_iters=32)` (encoders + correlation build + 32 RAFT
iterations) on a batch of synthetic N=8192 cloud pairs with seeded random-init weights.
value = sample-iterations/s = global_batch * iters / T_forward (CUDA events, max over ranks).
Rank 0 prints ONE JSON line.  See DESIGN.md "Measurement" for every field.

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (float32, float64 kept), so that two builds
can be compared output for output on identical seeded inputs:
  inference   flows.npy [iters, B, N, 3] (RSF: the flow of every iteration) or flow.npy [B, N, 3] (RSF_refine), whole batch
  training    loss.npy (rank 0's loss) and param.<name>.npy (every parameter after the step's Adam update)
  reference   flows.npy [32, 1, N, 3] of the last CPU forward
At most 64 MiB in all: a larger flow array keeps the same fixed, seeded sample of points in every sample and iteration.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_POINTS, TRUNC_K, ITERS, LEVELS, BASE_SCALE = 8192, 512, 32, 3, 0.25
BATCH_PER_GPU = 8        # 8 x 32 MiB of (corr, index) state = 268 MB > the 126 MB L2: the lookup streams from HBM
DUMP_LIMIT = 64 * 2 ** 20


def point_sample(t, limit=DUMP_LIMIT):
    """t [..., N, 3] of float32 cut to at most `limit` bytes: the same seeded subset of the N points (ascending) for every
    leading index, fixed by N and the size of t alone."""
    if t.numel() * 4 <= limit:
        return t
    n = t.shape[-2]
    keep = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:n * limit // (t.numel() * 4)].sort().values
    return t.index_select(-2, keep.to(t.device))


def dump_outputs(directory, arrays):
    """Write every array of `arrays` (name -> tensor) as <directory>/<name>.npy: float64 stays float64, the rest is float32."""
    host = {name: t.detach().cpu() for name, t in arrays.items()}
    host = {name: (t if t.dtype == torch.float64 else t.float()).numpy() for name, t in host.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT:
        raise ValueError(f'--dump-outputs: {total} bytes exceed the {DUMP_LIMIT} byte limit')
    os.makedirs(directory, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(directory, f'{name}.npy'), a)


def alg_bytes_lookup(n, k, levels=LEVELS, bf16=False):
    """ALGORITHMIC bytes of one sample-iteration of the lookup kernel (SURVEY.md 8d):
    fp32: K*(4 B corr + 4 B index) + 12 B coords in, levels*27*4 B voxel means + 32*16 B kNN vectors out = N*4944;
    bf16 mode: K*(2 + 2) + 12 in, levels*27*2 + 32*8 out = N*2478."""
    if bf16:
        return n * (k * 4 + 12 + levels * 27 * 2 + 32 * 8)
    return n * (k * 8 + 12 + levels * 27 * 4 + 32 * 16)


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        try:
            return json.load(open(path)), 'measured'
        except Exception:   # noqa: BLE001
            pass
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0}, 'fallback'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:   # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:   # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, flag in zip(names, f[3:7]):
                if flag.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': mx, 'samples': len(sm),
                'reasons': sorted(reasons)}


def make_args():
    return types.SimpleNamespace(corr_levels=LEVELS, base_scales=BASE_SCALE, truncate_k=TRUNC_K)


def synthetic_clouds(b, n, seed):
    g = torch.Generator().manual_seed(seed)
    pc1 = 10.0 * torch.rand(b, n, 3, generator=g)
    pc2 = pc1 + 0.1 * torch.randn(b, n, 3, generator=g)
    return pc1, pc2


# --------------------------------------------------------------------------------------------------
# CPU side: the reference's own formulation (oracle port, torch CPU ops) on the host cores
# --------------------------------------------------------------------------------------------------
_CPU_STATE = {}


def _cpu_weights():
    if 'W' not in _CPU_STATE:
        from pvraft_b200 import RSF
        torch.manual_seed(0)
        _CPU_STATE['W'] = {k: v.detach().clone() for k, v in RSF(make_args()).state_dict().items()}
    return _CPU_STATE['W']


def cpu_pick_threads():
    """torch CPU ops stop scaling (and then collapse) long before 100+ threads on these op sizes: time a
    small forward at a few thread counts and keep the fastest (reported as `cores`)."""
    if 'threads' in _CPU_STATE:
        return _CPU_STATE['threads']
    from oracle import pvraft_oracle as O
    W = _cpu_weights()
    pc1, pc2 = synthetic_clouds(1, 2048, 7)
    ncpu = os.cpu_count() or 1
    best, best_t = 1, float('inf')
    for th in sorted({t for t in (4, 8, 16, 32, 64, ncpu) if t <= ncpu}):
        torch.set_num_threads(th)
        with torch.no_grad():
            t0 = time.perf_counter()
            O.rsf_forward(W, pc1, pc2, 1, LEVELS, BASE_SCALE, TRUNC_K)
            t = time.perf_counter() - t0
        if t < best_t:
            best, best_t = th, t
    _CPU_STATE['threads'] = best
    return best


def cpu_sample(threads, loop_iters=ITERS, n=N_POINTS):
    """One CPU sample of the bench workload at B=1: everything before the loop (encoders, graphs, correlation build) +
    `loop_iters` RAFT iterations (all 32 by default: nothing is extrapolated), timed separately.
    Returns (t_prepare, t_loop, the flow of every iteration)."""
    from oracle import pvraft_oracle as O
    W = _cpu_weights()
    torch.set_num_threads(threads)
    pc1, pc2 = synthetic_clouds(1, n, 1234)
    with torch.no_grad():
        t0 = time.perf_counter()
        li = O.prepare(W, pc1, pc2, TRUNC_K)
        t1 = time.perf_counter()
        flows = O.raft_loop(W, li, pc1, loop_iters, LEVELS, BASE_SCALE)
        t2 = time.perf_counter()
    return t1 - t0, t2 - t1, flows


def gpu_reference_sample(dev, batch, iters):
    """The reference FORMULATION on the same GPU: the oracle's op sequence (= the reference's own ATen ops, model/*.py) run by
    torch eager on `dev`, fp32, TF32 off -- "the reference GPU build" of BASELINE.json's >= 10x target (the unmodified
    reference cannot travel to the GPU box).  One warm-up at 2 iterations, one timed forward; returns seconds."""
    from oracle import pvraft_oracle as O
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        W = {k: v.to(dev) for k, v in _cpu_weights().items()}
        pc1, pc2 = [t.to(dev) for t in synthetic_clouds(batch, N_POINTS, 1234)]
        with torch.no_grad():
            O.rsf_forward(W, pc1, pc2, 2, LEVELS, BASE_SCALE, TRUNC_K)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            O.rsf_forward(W, pc1, pc2, iters, LEVELS, BASE_SCALE, TRUNC_K)
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
        torch.cuda.empty_cache()


def gpu_reference_train_sample(dev, batch, iters):
    """One training step (forward + backward through torch autograd + Adam) of the reference's op sequence on `dev`, as
    gpu_reference_sample: fp32, TF32 off, one warm-up step then one timed step; returns seconds."""
    from oracle import pvraft_oracle as O
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        W = {k: v.to(dev).requires_grad_(True) for k, v in _cpu_weights().items()}
        opt = torch.optim.Adam(list(W.values()), lr=1e-3)
        pc1, pc2 = [t.to(dev) for t in synthetic_clouds(batch, N_POINTS, 1234)]

        def step():
            opt.zero_grad(set_to_none=True)
            flows = O.rsf_forward(W, pc1, pc2, iters, LEVELS, BASE_SCALE, TRUNC_K)
            n = len(flows)
            sum(0.8 ** (n - i - 1) * (flows[i] - (pc2 - pc1)).abs().sum(-1).mean() for i in range(n)).backward()
            opt.step()

        step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
        torch.cuda.empty_cache()


def run_reference(a):
    """`--impl reference`: the reference's CPU formulation (oracle port; the reference itself is pure PyTorch and is not present on
    the GPU box) timed on the host cores, same metric / unit / config.  A step is ONE full forward at B=1: the pre-loop work
    and all 32 iterations are executed and timed (no extrapolation), --steps of them (each takes tens of seconds)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return None
    threads = cpu_pick_threads()
    warm = min(a.warmup, 1)
    for _ in range(warm):
        cpu_sample(threads, 1)
    t_prep = t_loop = 0.0
    done = a.steps
    for _ in range(done):
        tp, tl, flows = cpu_sample(threads)
        t_prep += tp
        t_loop += tl
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {'flows': point_sample(torch.stack(flows))})
    t_prep /= done
    t_loop /= done
    value = ITERS / (t_prep + t_loop)
    line = {
        'impl': 'reference', 'metric': 'raft_sample_iters_per_sec', 'value': value, 'unit': 'sample-iterations/s',
        'n_gpus': a.gpus, 'steps': done, 'warmup': warm, 'ms_per_step': 1e3 * (t_prep + t_loop),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(1, 1, ITERS),
        'cpu_baseline': {'value': value, 'unit': 'sample-iterations/s', 'cores': threads, 'kind': 'port',
                         'sample': f'{done} full forwards at B=1, N={N_POINTS} (pre-loop work + all {ITERS} RAFT iterations, each '
                                   f'measured: t_prepare={t_prep:.2f} s, t_loop={t_loop:.2f} s); torch CPU ops, '
                                   f'{threads} of {os.cpu_count()} host threads (fastest of a thread sweep)'},
        'e2e': {'value': value, 'unit': 'sample-iterations/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    return line


def workload_config(batch_per_gpu, world, iters, graph=False, refine=False, dtype='f32'):
    state_mb = batch_per_gpu * N_POINTS * TRUNC_K * (4 if dtype == 'bf16' else 8) / 1e6
    l2 = (f'per-iteration candidate state ({state_mb:.0f} MB/GPU) exceeds the 126 MB L2; no explicit flush' if state_mb > 126
          else f'per-iteration candidate state is {state_mb:.0f} MB/GPU: L2-resident after the first iteration (labelled as such)')
    mode = ('bf16 correlation state + uint16 ids, fp32 coordinates / index math / layers (BASELINE.json configs[2])' if dtype == 'bf16'
            else 'fp32 (BASELINE.json metric config; batch from configs[2])')
    return {'workload': f'{"RSF_refine" if refine else "RSF"}.forward: N={N_POINTS} pts x2 clouds, truncate_k={TRUNC_K}, corr_levels={LEVELS}, '
                        f'iters={iters}, batch {batch_per_gpu}/GPU, {mode}'
                        + (', CUDA-graph replay' if graph else ''),
            'global_batch': batch_per_gpu * world, 'points': N_POINTS, 'truncate_k': TRUNC_K, 'iters': iters,
            'parallelism': f'batch-shard x{world} (no data-path collective)', 'l2_policy': l2}


def lookup_traffic():
    """dram__bytes_read+write per launch of the lookup kernel from the committed ncu capture -- only while that capture
    belongs to the kernel source that is being timed (profiles/lookup_dram_bytes.json records the source's sha256)."""
    import hashlib
    path = os.path.join(ROOT, 'profiles', 'lookup_dram_bytes.json')
    src = os.path.join(ROOT, 'pvraft_b200', 'csrc', 'corr_lookup.cu')
    try:
        rec = json.load(open(path))
        if rec.get('source_sha256') == hashlib.sha256(open(src, 'rb').read()).hexdigest():
            return rec.get('dram_bytes_per_launch')
    except Exception:   # noqa: BLE001
        pass
    return None


# --------------------------------------------------------------------------------------------------
# native arm
# --------------------------------------------------------------------------------------------------
def run_native(a):
    from pvraft_b200 import RSF, RSF_refine, ops
    from pvraft_b200 import dist as D
    rank, world, local = D.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    B, iters = a.batch, a.iters
    torch.manual_seed(0)
    model = (RSF_refine if a.refine else RSF)(make_args()).to(dev).eval()
    model.set_precision('bf16' if a.dtype == 'bf16' else 'fp32')
    last = (lambda out: out) if a.refine else (lambda out: out[-1])
    if a.graph is not None:
        model.use_cuda_graph = bool(a.graph)
    # default policy of the model: graph replay from the first call for B <= 2, from the second call with the same shape and
    # unchanged weights otherwise -- the warm-up steps put every timed step on the replay path
    graphed = model.use_cuda_graph if model.use_cuda_graph is not None else True
    pc1_h, pc2_h = synthetic_clouds(B, N_POINTS, 1234 + rank)
    pc1_h, pc2_h = pc1_h.pin_memory(), pc2_h.pin_memory()
    pc1, pc2 = pc1_h.to(dev), pc2_h.to(dev)
    out_h = torch.empty(B, N_POINTS, 3).pin_memory()
    result = [None]      # what the latest resident step returned (--dump-outputs)

    def step_resident():
        with torch.no_grad():
            result[0] = model([pc1, pc2], iters)

    def step_e2e():
        with torch.no_grad():
            flow = last(model([pc1_h.to(dev, non_blocking=True), pc2_h.to(dev, non_blocking=True)], iters))
            out_h.copy_(flow, non_blocking=True)
        return flow

    def timed(fn, steps, sample_clocks=False):
        D.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local) if sample_clocks and rank == 0 else None
        if sampler:
            sampler.start()
        l0 = ops.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        D.barrier()
        ms = D.max_over_ranks(e0.elapsed_time(e1), dev)
        clocks = sampler.stop() if sampler else None
        return ms, ops.launch_count - l0, clocks

    for _ in range(max(a.warmup, 3)):
        step_resident()
    ms, launches, clocks = timed(step_resident, a.steps, sample_clocks=True)
    if clocks and set(clocks['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}:
        ms, launches, clocks = timed(step_resident, a.steps, sample_clocks=True)     # re-measure once
    if a.dump_outputs:
        if a.refine:
            outputs = {'flow': point_sample(D.gather_batch(result[0]))}
        else:
            outputs = {'flows': point_sample(torch.stack([D.gather_batch(f) for f in result[0]]))}
        if rank == 0:
            dump_outputs(a.dump_outputs, outputs)
    step_e2e()
    ms_e2e, _, _ = timed(step_e2e, a.steps)
    gb = B * world
    value = gb * iters * a.steps / (ms * 1e-3)
    e2e = gb * iters * a.steps / (ms_e2e * 1e-3)

    # ---- dominant kernel: the fused correlation lookup, timed in situ with CUDA events ----------------
    lk_ms = []
    orig = ops.corr_lookup

    def hooked(*args, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        r = orig(*args, **kw)
        e.record()
        lk_ms.append((s, e))
        return r

    ops.corr_lookup = hooked
    was_graph = model.use_cuda_graph
    model.use_cuda_graph = False            # per-launch events need the eager launch sequence
    for _ in range(3):
        step_resident()
    torch.cuda.synchronize()
    ops.corr_lookup = orig
    model.use_cuda_graph = was_graph
    # the first eager step starts on an empty queue (the timed steps were graph replays): until the host is ahead of the GPU an
    # event pair also spans the host's launch latency, so that step's pairs are dropped
    lk_ms = lk_ms[len(lk_ms) // 3:]
    durs = [s.elapsed_time(e) for s, e in lk_ms]
    lookup_ms = statistics.mean(durs)
    peaks, peak_kind = measured_peaks()
    alg = alg_bytes_lookup(N_POINTS, TRUNC_K, bf16=a.dtype == 'bf16') * B
    achieved = alg / (lookup_ms * 1e-3) / 1e9
    roofline = {'kernel': 'k_corr_lookup (pvraft_corr_lookup_bf16_fwd)' if a.dtype == 'bf16' else 'k_corr_lookup (pvraft_corr_lookup_fwd)', 'bound': 'hbm', 'achieved': achieved,
                'peak': peaks['hbm_gbs'], 'peak_kind': peak_kind + ' (MEASURED_PEAKS.json hbm_gbs)' if peak_kind == 'measured' else 'fallback',
                'unit': 'GB/s', 'frac': achieved / peaks['hbm_gbs'], 'traffic': lookup_traffic() if a.dtype == 'f32' else None,
                'alg_bytes_per_launch': alg, 'avg_launch_ms': lookup_ms, 'launches_timed': len(durs),
                'share_of_step': lookup_ms * iters / (ms / a.steps)}

    if rank != 0:
        return None
    cpu = gpu_ref = None

    def assemble():
        return {
            'metric': 'raft_sample_iters_per_sec', 'value': value, 'unit': 'sample-iterations/s', 'n_gpus': world,
            'steps': a.steps, 'warmup': max(a.warmup, 3), 'ms_per_step': ms / a.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': a.dtype, 'data': 'synthetic',
            'config': workload_config(B, world, iters, graphed, a.refine, a.dtype),
            'e2e': {'value': e2e, 'unit': 'sample-iterations/s', 'h2d_bytes_per_step': 2 * B * N_POINTS * 3 * 4 * world,
                    'd2h_bytes_per_step': B * N_POINTS * 3 * 4 * world, 'ms_per_step': ms_e2e / a.steps},
            'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline, 'cpu_baseline': cpu, 'gpu_reference': gpu_ref,
        }

    # The measurement proper is complete here.  The two baseline legs below run foreign code (torch CPU / torch eager ops of
    # the oracle) for ~25 s and ~2 s; if one of them ever stalls (an oversubscribed host, a wedged OpenMP team), the line is
    # still printed -- with that leg marked unavailable -- instead of the whole run being lost.
    legs_done = threading.Event()

    def watchdog(limit_s=float(os.environ.get('PVRAFT_BENCH_LEG_LIMIT', '420'))):
        if legs_done.wait(limit_s):
            return
        nonlocal cpu, gpu_ref
        note = {'unavailable': f'baseline leg did not finish within {limit_s:.0f} s'}
        cpu = cpu if cpu is not None else dict(note, value=None, unit='sample-iterations/s', cores=None, kind='port', sample='none')
        gpu_ref = gpu_ref if gpu_ref is not None else note
        _emit_and_exit(assemble())

    if world == 1 and not (a.no_cpu and (a.no_gpu_ref or a.refine)):
        threading.Thread(target=watchdog, daemon=True).start()
    if world == 1 and not a.no_cpu:
        threads = cpu_pick_threads()
        tp, tl, _ = cpu_sample(threads)
        cpu = {'value': ITERS / (tp + tl), 'unit': 'sample-iterations/s', 'cores': threads, 'kind': 'port',
               'sample': f'one full forward at B=1, N={N_POINTS}: pre-loop work + all {ITERS} RAFT iterations, measured '
                         f'(t_prepare={tp:.2f} s, t_loop={tl:.2f} s; oracle port of the reference, torch CPU ops, '
                         f'{threads} of {os.cpu_count()} host threads)'}
    if world == 1 and not a.no_gpu_ref and not a.refine:
        try:
            t_ref = gpu_reference_sample(dev, B, iters)
            gpu_ref = {'value': B * iters / t_ref, 'unit': 'sample-iterations/s', 'ms_per_step': 1e3 * t_ref,
                       'kind': "the reference's own op sequence (oracle port of model/*.py) in torch eager on this GPU, fp32, TF32 off, "
                               f'batch {B}, {iters} iterations, one timed forward after a warm-up',
                       'speedup': value / (B * iters / t_ref)}
        except Exception as e:   # noqa: BLE001  (out of memory on a smaller device: report, do not fail the bench)
            gpu_ref = {'unavailable': f'{type(e).__name__}: {e}'[:200]}
    legs_done.set()
    line = assemble()
    return line


# --------------------------------------------------------------------------------------------------
# training step (BASELINE.json configs[3]): fwd + bwd + Adam, batch sharded over the ranks, ONE gradient all-reduce
# --------------------------------------------------------------------------------------------------
def run_train(a):
    import torch.distributed as dist
    from pvraft_b200 import RSF, ops
    from pvraft_b200 import dist as D
    rank, world, local = D.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    B, iters = a.batch, a.iters
    torch.manual_seed(0)
    model = RSF(make_args()).to(dev).train()
    wrapped = D.ddp(model, local)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)                       # tools/engine.py:57
    pc1_h, pc2_h = synthetic_clouds(B, N_POINTS, 1234 + rank)
    pc1_h, pc2_h = pc1_h.pin_memory(), pc2_h.pin_memory()
    pc1, pc2 = pc1_h.to(dev), pc2_h.to(dev)
    loss_h = torch.empty(1).pin_memory()
    last_loss = [None]   # the latest step's loss (under graph replay: the captured step's, refreshed by every replay)

    def loss_fn(flows, gt, gamma=0.8):                                        # tools/loss.py:4-13 (all-ones mask)
        n = len(flows)
        return sum(gamma ** (n - i - 1) * (flows[i] - gt).abs().sum(-1).mean() for i in range(n))

    def step(x1, x2):
        opt.zero_grad(set_to_none=True)
        flows = wrapped([x1, x2], num_iters=iters)
        loss = loss_fn(flows, x2 - x1)
        loss.backward()                                                       # DDP: the 750 KiB gradient all-reduce happens here
        opt.step()
        last_loss[0] = loss.detach()
        return loss

    def step_resident():
        return step(pc1, pc2)

    def step_e2e():
        loss = step(pc1_h.to(dev, non_blocking=True), pc2_h.to(dev, non_blocking=True))
        loss_h.copy_(loss.detach().reshape(1), non_blocking=True)
        return loss

    def timed(fn, steps):
        D.barrier()
        torch.cuda.synchronize()
        l0 = ops.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        D.barrier()
        return D.max_over_ranks(e0.elapsed_time(e1), dev), ops.launch_count - l0

    for _ in range(max(a.warmup, 3)):
        step_resident()
    graphed = False
    if a.graph and world == 1:
        # whole-step CUDA graph (forward + backward + Adam): the eager step is bound by the host launch path (~660 library
        # launches + ATen glue per step); replaying one graph shows what the kernels themselves take
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(3):
                step_resident()
        torch.cuda.current_stream(dev).wait_stream(side)
        launches_per_step = [0]
        g = torch.cuda.CUDAGraph()
        l0 = ops.launch_count
        with torch.cuda.graph(g):
            step_resident()
        launches_per_step[0] = ops.launch_count - l0

        def step_resident():   # noqa: F811
            g.replay()
            ops.launch_count += launches_per_step[0]

        def step_e2e():   # noqa: F811
            pc1.copy_(pc1_h, non_blocking=True)
            pc2.copy_(pc2_h, non_blocking=True)
            step_resident()
        graphed = True
        for _ in range(3):
            step_resident()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches = timed(step_resident, a.steps)
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, dict({'loss': last_loss[0]}, **{f'param.{k}': p for k, p in model.named_parameters()}))
    ms_e2e, _ = timed(step_e2e, a.steps)
    # the collective alone: one all-reduce of a gradient-sized fp32 buffer
    nparam = sum(p.numel() for p in model.parameters())
    coll = {'bytes': nparam * 4, 'ranks': world, 'standalone_us': None}
    if world > 1:
        buf = torch.zeros(nparam, device=dev)
        for _ in range(5):
            dist.all_reduce(buf)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            dist.all_reduce(buf)
        e1.record()
        torch.cuda.synchronize()
        coll['standalone_us'] = D.max_over_ranks(e0.elapsed_time(e1) / 20 * 1e3, dev)
        coll['share_of_step'] = coll['standalone_us'] * 1e-3 / (ms / a.steps)
    if rank != 0:
        return None
    gb = B * world
    gpu_ref = None
    if world == 1 and not a.no_gpu_ref:
        try:
            t_ref = gpu_reference_train_sample(dev, B, iters)
            gpu_ref = {'value': B * iters / t_ref, 'unit': 'sample-iterations/s', 'ms_per_step': 1e3 * t_ref,
                       'kind': "the reference's own op sequence (oracle port of model/*.py) with torch autograd + Adam in torch eager "
                               f'on this GPU, fp32, TF32 off, batch {B}, {iters} iterations, one timed step after a warm-up step',
                       'speedup': (gb * iters * a.steps / (ms * 1e-3)) / (B * iters / t_ref)}
        except Exception as e:   # noqa: BLE001
            gpu_ref = {'unavailable': f'{type(e).__name__}: {e}'[:200]}
    return {
        'metric': 'raft_train_sample_iters_per_sec', 'value': gb * iters * a.steps / (ms * 1e-3), 'unit': 'sample-iterations/s',
        'n_gpus': world, 'steps': a.steps, 'warmup': max(a.warmup, 3), 'ms_per_step': ms / a.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'training step (forward + backward + Adam) of RSF: N={N_POINTS} pts x2 clouds, truncate_k={TRUNC_K}, '
                               f'iters={iters}, batch {B}/GPU, fp32 (BASELINE.json configs[3])' + (', whole step replayed as one CUDA graph' if graphed else ''),
                   'global_batch': gb, 'points': N_POINTS,
                   'truncate_k': TRUNC_K, 'iters': iters,
                   'parallelism': f'DDP batch-shard x{world}: one gradient all-reduce of {nparam * 4} B per step (NCCL)'},
        'e2e': {'value': gb * iters * a.steps / (ms_e2e * 1e-3), 'unit': 'sample-iterations/s',
                'h2d_bytes_per_step': 2 * B * N_POINTS * 3 * 4 * world, 'd2h_bytes_per_step': 4 * world, 'ms_per_step': ms_e2e / a.steps},
        'gpu_launches': launches, 'clocks': clocks, 'collective': coll, 'gpu_reference': gpu_ref,
    }


_SAVED_STDOUT = [None]


def _emit_and_exit(line):
    """Print the JSON line on the real stdout (fd 1 is routed to stderr while the benchmark runs) and leave."""
    fd = _SAVED_STDOUT[0] if _SAVED_STDOUT[0] is not None else 1
    os.write(fd, (json.dumps(line) + '\n').encode())
    os._exit(0)


class _QuietStdout:
    """Libraries (NCCL's version banner, warnings) write to fd 1; the contract is ONE JSON line on stdout.
    Route fd 1 to stderr while the benchmark runs and restore it for the final print."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        _SAVED_STDOUT[0] = self.saved
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        _SAVED_STDOUT[0] = None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=40)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', choices=['native', 'reference'], default='native')
    ap.add_argument('--mode', choices=['infer', 'train'], default='infer', help='train = BASELINE configs[3] (fwd+bwd+Adam, DDP)')
    ap.add_argument('--batch', type=int, default=None, help='samples per GPU (default 8; 2 in train mode)')
    ap.add_argument('--iters', type=int, default=None, help='RAFT iterations (default 32; 8 in train mode)')
    ap.add_argument('--graph', type=int, default=None, help='1/0 force CUDA-graph replay on/off (default: automatic for batch <= 2)')
    ap.add_argument('--dtype', choices=['f32', 'bf16'], default='f32', help='bf16 = reduced-precision correlation state (configs[2])')
    ap.add_argument('--refine', action='store_true', help='RSF_refine instead of RSF (configs[2])')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-gpu-ref', action='store_true', help='skip the gpu_reference leg')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (at most 64 MiB; see the module's docstring)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.batch is None:
        a.batch = 2 if a.mode == 'train' else BATCH_PER_GPU
    if a.iters is None:
        a.iters = 8 if a.mode == 'train' else ITERS
    with _QuietStdout():
        if a.impl == 'reference':
            line = run_reference(a)
        else:
            line = run_train(a) if a.mode == 'train' else run_native(a)
    if line is not None:
        print(json.dumps(line), flush=True)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
