#!/usr/bin/env python
"""bench.py - image-pairs/sec of the OpenGlue matching core on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload C3] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one pass of the whole hot path (keypoint encoder -> 18 attention layers -> score
matrix -> 100 Sinkhorn iterations -> mutual matches) over one batch of synthetic image pairs per
GPU (weak scaling: per-GPU batch fixed, pairs are independent, no data-path collective; one tiny
NCCL all-reduce of the per-rank match statistics per step mirrors the reference's
`self.log(..., sync_dist=True)`).

Prints ONE JSON line (rank 0).  Keys follow the driver's contract; `roofline` is measured live
on the dominant kernel through the operator-level C-ABI call, `cpu_baseline` / `--impl reference`
time the unmodified reference module staged under oracle/_ref (oracle/build_ref.py; `kind: "reference"`) on the host
cores, or - when it is not staged - the oracle port (same ATen ops, bit-identical outputs; `kind: "port"`).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark runs from the built tree and writes nothing into it

import torch  # noqa: E402

from openglue_b200.synthetic import BASELINE_CONFIGS, default_config, synthetic_pairs, synthetic_state_dict  # noqa: E402

METRIC = 'image-pairs/sec at N=M=2048, d=256, 9 GNN layers, 100 Sinkhorn iters'
MATCH_THRESHOLD = 0.2
DUMP_BYTES = 60 << 20               # --dump-outputs writes less than 64 MB in all, .npy headers included


def flops_per_pair(n, m, d, stages, s):
    """SURVEY.md section 8(d) / BASELINE.md section 4 (multiply-add = 2 FLOP, exp not counted)."""
    f_attn = 4 * d * stages * (n + m) ** 2
    f_lin = 40 * stages * (n + m) * d * d
    f_final = 2 * (n + m) * d * d + 2 * n * m * d
    f_pe = 2 * (n + m) * (32 * (2 + s) + 32 * 64 + 64 * 128 + 128 * d)
    return dict(total=f_attn + f_lin + f_final + f_pe, attn=f_attn, lin=f_lin)


def sinkhorn_bytes_per_pair(n, m, iters):
    return (iters + 1) * 4 * (n + 1) * (m + 1)


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p['hbm_gbs'], bf16_tflops=p['bf16_tflops'],
                    bf16_tflops_sustained=p.get('bf16_tflops_sustained', p['bf16_tflops']), source='measured')
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source='fallback')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,' \
        'clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile('w', suffix='.csv', delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            parts = [x.strip() for x in line.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), parts[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        busy = sorted(sm)[len(sm) // 2:]                      # upper half = samples under load
        return {'sm_mhz': statistics.median(busy), 'sm_max_mhz': max(mx), 'reasons': sorted(reasons), 'samples': len(sm)}


def verify_against_fixture(args, res, batch, rank):
    """The output of the timed configuration against the fixture minted from the unmodified reference for exactly these inputs
    (tests/golden/<workload>_planted.pt: synthetic_pairs(batch, seed=1234) = rank 0's batch).  A mismatch is an error, not a
    footnote: a fast wrong answer is not a result."""
    path = os.path.join(ROOT, 'tests', 'golden', f'{args.workload}_planted.pt')
    if rank != 0 or not os.path.exists(path):
        return None
    fx = torch.load(path, weights_only=False)
    if fx['batch'] != batch:
        return {'fixture': os.path.basename(path), 'skipped': f'fixture batch {fx["batch"]} != {batch}'}
    m0, ms0 = res['matches0'].cpu(), res['matching_scores0'].cpu()
    mism = int((m0 != fx['matches0']).sum())
    err = float((ms0 - fx['matching_scores0']).abs().max())
    out = {'fixture': os.path.basename(path), 'pairs': batch, 'matches0_identical': mism == 0, 'matches0_mismatches': mism,
           'matches': int((m0 >= 0).sum()), 'max_abs_matching_score_err': err,
           'reference': 'MatchingTrainingModule.forward of the unmodified reference, fp32 CPU (oracle/gen_golden.py)'}
    if mism != 0 or err > 3e-4:
        raise SystemExit('bench.py: the timed output does not match the reference fixture: ' + json.dumps(out))
    return out


def dump_outputs(out_dir, arrays):
    """--dump-outputs: one <out_dir>/<name>.npy per array, float32 kept as float32 and every other dtype stored as float64 (exact
    for the match indices), so that two builds can be compared output for output on identical inputs.  An array larger than its
    share of DUMP_BYTES is stored as a fixed sample: its flattened elements at indices drawn by a generator seeded with 0 (sorted,
    duplicates dropped), with those indices in <name>_sample_index.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        t = t.detach()
        t = t if t.dtype == torch.float32 else t.double()
        if t.numel() * t.element_size() > share:
            idx = torch.randint(t.numel(), (share // 16,), generator=torch.Generator().manual_seed(0)).unique()
            np.save(os.path.join(out_dir, f'{name}_sample_index.npy'), idx.double().numpy())
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, f'{name}.npy'), t.cpu().numpy())


def _numa_nodes():
    """CPU lists of the NUMA nodes (Linux sysfs); one pseudo-node with every CPU if unavailable."""
    nodes = []
    try:
        base = '/sys/devices/system/node'
        for name in sorted(os.listdir(base)):
            if name.startswith('node') and name[4:].isdigit():
                cpus = []
                for part in open(os.path.join(base, name, 'cpulist')).read().strip().split(','):
                    lo, _, hi = part.partition('-')
                    cpus += list(range(int(lo), int(hi or lo) + 1))
                if cpus:
                    nodes.append(cpus)
    except OSError:
        pass
    allowed = sorted(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else list(range(os.cpu_count() or 8))
    nodes = [[c for c in n if c in allowed] for n in nodes]
    nodes = [n for n in nodes if n]
    return nodes or [allowed]


def _reference_kind():
    """'reference' when the unmodified reference is staged under oracle/_ref (oracle/build_ref.py; it travels to the GPU box),
    else 'port' (the oracle restatement: the same ATen calls, bit-identical outputs - tests/test_oracle_golden.py)."""
    from oracle.build_ref import available
    return 'reference' if available() else 'port'


def _oracle_times(cfg, n, m, reps, threads, family='planted'):
    from oracle import superglue_oracle as O                  # checker / CPU baseline only
    from oracle.build_ref import import_reference
    sd = synthetic_state_dict(cfg, seed=0)
    data = synthetic_pairs(1, n, m, cfg['descriptor_dim'], cfg['positional_encoding']['side_info_size'], family=family, seed=1234)
    torch.set_num_threads(threads)
    ref = import_reference()
    if ref is not None:                                       # the reference's own module + the match extraction of matching_module.py:175-181
        model = ref[0](dict(cfg)).eval()
        model.load_state_dict(sd)

        def run():
            with torch.no_grad():
                return O.extract_matches(model(data)['scores'], MATCH_THRESHOLD)
    else:
        def run():
            return O.run(sd, cfg, data, MATCH_THRESHOLD)
    run()                                                     # warm-up at this thread count
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        run()
        times.append(time.perf_counter() - t0)
    return times


def cpu_worker(argv):
    """internal: `bench.py --cpu-worker WORKLOAD REPS THREADS cpu,cpu,...` - one pinned process of the multi-process CPU baseline"""
    wl = BASELINE_CONFIGS[argv[0]]
    reps, threads = int(argv[1]), int(argv[2])
    os.sched_setaffinity(0, {int(c) for c in argv[3].split(',')})
    times = _oracle_times(default_config(**wl['cfg']), wl['n'], wl['m'], reps, threads)
    print(json.dumps({'times': times}), flush=True)


def time_oracle(workload, cfg, n, m, reps):
    """The CPU path of the reference (oracle port: same ATen ops), one pair per run, on this box's host cores.
    (a) ONE process pinned to one NUMA node (an unpinned process on a 2-socket host pays remote-memory traffic: round 1 measured
        0.32 pairs/s unpinned against 0.5-0.6 on 8 local cores), intra-op thread count swept, best kept;
    (b) the AGGREGATE of several such processes side by side, each pinned to its own slice of cores - what the host can do for this
        embarrassingly parallel job with all its cores.
    Returns dict(single=pairs/s, threads=..., aggregate=pairs/s, procs=..., cores=...)."""
    nodes = _numa_nodes()
    node0 = nodes[0]
    default_threads = torch.get_num_threads()
    old_aff = os.sched_getaffinity(0) if hasattr(os, 'sched_getaffinity') else None
    out = {'numa_nodes': len(nodes), 'cpus': sum(len(x) for x in nodes)}
    try:
        if old_aff is not None:
            os.sched_setaffinity(0, set(node0))
        best_t, best = 1, float('inf')
        for t in sorted({t for t in (8, 16, 32, min(64, len(node0))) if t <= len(node0)}):       # (64+ threads: 0.08 pairs/s in round 1; the sweep stops at the first count that is 2x slower than the best)
            dt = min(_oracle_times(cfg, n, m, 1, t))
            if dt < best:
                best_t, best = t, dt
            if dt > 2 * best:
                break
        times = _oracle_times(cfg, n, m, reps, best_t)
        out.update(single=1.0 / min(times), single_mean=len(times) / sum(times), threads=best_t, node0_cpus=len(node0), times=times)
    finally:
        if old_aff is not None:
            os.sched_setaffinity(0, old_aff)
        torch.set_num_threads(default_threads)
    # (b) side-by-side processes: slices of `per` cores inside each NUMA node
    per = min(16, len(node0))
    slices = [node[i:i + per] for node in nodes for i in range(0, len(node) - per + 1, per)]
    procs = []
    t0 = time.perf_counter()
    for sl in slices:
        # one warm-up + ONE timed pair per process: with every core busy a pair takes ~30 s on the GPU box's host (memory-bound), and
        # this leg only has to show that more processes do not beat the single pinned one (visit Y: the default run took 200 s)
        cmd = [sys.executable, os.path.abspath(__file__), '--cpu-worker', workload, '1', str(per), ','.join(map(str, sl))]
        env = dict(os.environ, OMP_NUM_THREADS=str(per), MKL_NUM_THREADS=str(per))
        procs.append(subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=env))
    rates = []
    for pr in procs:
        try:
            so, _ = pr.communicate(timeout=600)
            tt = json.loads(so.strip().splitlines()[-1])['times']
            rates.append(len(tt) / sum(tt))                   # steady-state rate of this process while its neighbours run
        except Exception:
            pr.kill()
    out.update(aggregate=sum(rates), procs=len(rates), cores_per_proc=per, aggregate_wall_s=time.perf_counter() - t0)
    return out


def run_reference(args, wl):
    """--impl reference: the reference's own CPU implementation of the path on the host cores: the unmodified reference module
    staged under oracle/_ref by oracle/build_ref.py (kind "reference"), else the oracle port (kind "port")."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cfg = default_config(**wl['cfg'])
    # each step = a bounded sample of the workload: ONE pair of the workload's shape per process
    r = time_oracle(args.workload, cfg, wl['n'], wl['m'], max(1, args.steps))
    value = max(r['single'], r.get('aggregate', 0.0))         # all the host threads it can use
    cores = r['procs'] * r['cores_per_proc'] if r.get('aggregate', 0.0) >= r['single'] else r['threads']
    kind = _reference_kind()
    what = 'the unmodified reference SuperGlue module from oracle/_ref + its match extraction' if kind == 'reference' else 'oracle port = the reference\'s ATen ops'
    sample = (f'1 pair per step of the {args.workload} shape (N={wl["n"]}, M={wl["m"]}), torch CPU fp32 ({what}); '
              f'single process pinned to NUMA node 0 ({r["node0_cpus"]} cpus), {r["threads"]} threads (best of a sweep): {r["single"]:.3f} pairs/s; '
              f'{r["procs"]} processes side by side x {r["cores_per_proc"]} pinned cores: {r.get("aggregate", 0.0):.3f} pairs/s aggregate; '
              f'value = the larger; host: {r["cpus"]} cpus, {r["numa_nodes"]} NUMA nodes')
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'pairs/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': 1, 'ms_per_step': 1e3 / value, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': bench_config(args, wl, per_gpu_batch=1),
        'cpu_baseline': {'value': value, 'unit': 'pairs/s', 'cores': cores, 'kind': kind, 'sample': sample,
                         'single_process': r['single'], 'aggregate': r.get('aggregate')},
        'e2e': {'value': value, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def bench_config(args, wl, per_gpu_batch):
    c = wl['cfg']
    return {'workload': f'{args.workload}: {per_gpu_batch} pairs/GPU, N={wl["n"]}, M={wl["m"]}, d={c["descriptor_dim"]}, '
                        f'{c["num_stages"]} stages (self+cross), {c["num_iters"]} Sinkhorn iters, planted synthetic pairs',
            'pairs_per_gpu': per_gpu_batch, 'global_pairs': per_gpu_batch * args.gpus,
            'N': wl['n'], 'M': wl['m'], 'd': c['descriptor_dim'], 'stages': c['num_stages'],
            'sinkhorn_iters': c['num_iters'], 'parallelism': f'pairs sharded over {args.gpus} GPU(s), no data-path collective',
            'l2': 'working set per step (scores 16.8 MB/pair + activations) exceeds the 126 MB L2; no explicit flush',
            'cuda_graph': bool(getattr(args, 'cuda_graph', 0))}


def main():
    if len(sys.argv) > 1 and sys.argv[1] == '--cpu-worker':
        return cpu_worker(sys.argv[2:])
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=8)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='C3', choices=sorted(BASELINE_CONFIGS))
    ap.add_argument('--pairs-per-gpu', type=int, default=None)
    ap.add_argument('--precision', default=os.environ.get('OG_PRECISION', 'fp16x3'), choices=['fp32', 'tf32x3', 'fp16x3'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-verify', action='store_true', help='skip the check of the timed output against tests/golden/<workload>_planted.pt')
    ap.add_argument('--cuda-graph', type=int, default=1, help='replay the launch schedule from a CUDA graph (default on)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write rank 0's outputs of the last timed step as DIR/<name>.npy (float32 / float64, under 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    wl = dict(BASELINE_CONFIGS[args.workload])
    if args.impl == 'reference':
        return run_reference(args, wl)

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if world != args.gpus and world > 1:
        raise SystemExit(f'--gpus {args.gpus} but WORLD_SIZE={world}')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)

    from openglue_b200 import _cabi
    _cabi.lib()                                # the library build() left in the tree; a missing one is an error
    from openglue_b200.superglue import MatchingCore, SuperGlue

    batch = args.pairs_per_gpu or wl['batch']
    n, m = wl['n'], wl['m']
    cfg = default_config(**wl['cfg'])
    cfg['precision'] = args.precision
    d, s_dim, stages, iters = cfg['descriptor_dim'], cfg['positional_encoding']['side_info_size'], \
        cfg['attention_gnn']['num_stages'], cfg['otp']['num_iters']
    model = SuperGlue(cfg).eval()
    model.load_state_dict(synthetic_state_dict(cfg, seed=0))
    model = model.to(dev)
    core = MatchingCore(model, MATCH_THRESHOLD, device=dev, use_cuda_graph=bool(args.cuda_graph))
    host = synthetic_pairs(batch, n, m, d, s_dim, family='planted', seed=1234 + rank)
    host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in host.items()}
    data = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in host.items()}
    stats = torch.zeros(3, device=dev, dtype=torch.float64)
    loss_acc = torch.zeros(2, device=dev)

    from openglue_b200.sharding import all_reduce_loss, match_statistics
    with_loss = args.workload == 'C4'          # BASELINE.json configs[3]: reference criterion on every rank + NCCL loss all-reduce
    side = torch.cuda.Stream(dev)              # the collective runs beside the next step's kernels, never on the compute stream
    if with_loss:
        from openglue_b200 import generate_gt_matches
        from openglue_b200.losses import criterion
        # the planted similarity of synthetic_pairs (k1 = 0.9 k0 + 20) as the batch's ground-truth transformation: labels are
        # produced per step by og_gt_matches_fwd exactly as training_step does (matching_module.py:84-93)
        H = torch.tensor([[0.9, 0.0, 20.0], [0.0, 0.9, 20.0], [0.0, 0.0, 1.0]], device=dev).repeat(batch, 1, 1)
        transformation = {'type': ['perspective'] * batch, 'H': H}

    def reduce_on_side_stream(t, out):
        """sum over ranks of a small device tensor, on the side stream (self.log(..., sync_dist=True), matching_module.py:102-103)"""
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            if out is loss_acc:
                all_reduce_loss(t)                     # mean over ranks (sharding.py)
            elif dist is not None:
                dist.all_reduce(t)
            out.copy_(t)
        t.record_stream(side)

    def step(inputs):
        if with_loss and inputs is data:
            f0 = {'keypoints': inputs['keypoints0'], 'side_info': inputs['side_info0'], 'local_descriptors': inputs['local_descriptors0']}
            f1 = {'keypoints': inputs['keypoints1'], 'side_info': inputs['side_info1'], 'local_descriptors': inputs['local_descriptors1']}
            _, y_true = generate_gt_matches({'transformation': transformation}, f0, f1, 3.0, 5.0)
            res = core(inputs, want_scores=True, borrow=True)
            loss = criterion(y_true, res)
            reduce_on_side_stream(torch.stack([loss['loss'], loss['metric_loss']]), loss_acc)
            return res
        res = core(inputs, borrow=inputs is data)
        if dist is not None and inputs is data:   # the reference's sync_dist logging: one tiny NCCL all-reduce per step
            reduce_on_side_stream(match_statistics(res['matches0'], res['matching_scores0']), stats)
        return res

    def sync_all():
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(fn, steps):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- device-resident throughput (value) ----
    for _ in range(max(3, args.warmup)):
        step(data)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    last = {}
    ms_total = timed(lambda: last.update(step(data)), args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(last, loss=loss_acc) if with_loss else last)
    launches = model.last_launches * args.steps
    verified = verify_against_fixture(args, step(data), batch, rank) if not args.no_verify else None
    # ---- end to end through the public API with HOST buffers (H2D + D2H inside the timed region) ----
    for _ in range(2):
        step(host)
    ms_e2e_serial = timed(lambda: step(host), args.steps)          # blocking forward(): copy, compute, copy, in series

    # serving form of the same API: submit()/wait() with two batches in flight, so the upload of step i+1 overlaps
    # the kernels of step i; every step still uploads its inputs and reads its matches back inside the timed region
    def consume(res):
        if dist is not None:
            reduce_on_side_stream(match_statistics(res['matches0'], res['matching_scores0']).to(dev, non_blocking=True), stats)

    def pipelined(steps):
        pend = None
        for _ in range(steps):
            nxt = core.submit(host)
            if pend is not None:
                consume(pend.wait())
            pend = nxt
        consume(pend.wait())
    pipelined(2)
    ms_e2e = timed(lambda: pipelined(args.steps), 1)
    clocks = sampler.stop() if rank == 0 else None
    h2d = sum(v.numel() * v.element_size() for k, v in host.items() if torch.is_tensor(v) and k in core._TENSOR_KEYS)
    d2h = batch * (n * 8 + n * 4 + m * 8 + m * 4)

    ms_per_step = ms_total / args.steps
    value = batch * world / (ms_per_step * 1e-3)
    e2e_value = batch * world / (ms_e2e / args.steps * 1e-3)

    # ---- roofline of the dominant kernel: fused attention (self layer launch), measured live ----
    peaks = measured_peaks()
    lib = _cabi.lib()
    import ctypes as C
    H = cfg['attention_gnn']['num_heads']
    nb = 2 * batch if n == m else batch
    qkv = torch.randn(nb * n, 3 * d, device=dev)
    o = torch.empty(nb * n, d, device=dev)
    prec = {'fp32': _cabi.OG_PREC_FP32, 'tf32x3': _cabi.OG_PREC_TF32X3, 'fp16x3': _cabi.OG_PREC_FP16X3}[args.precision]
    p = lambda t, off=0: C.c_void_p(t.data_ptr() + off * 4)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    if args.precision == 'tf32x3' or (args.precision == 'fp16x3' and d // H != 64):    # head_dim 32 runs the tf32 form in either mode
        kk = torch.randn(nb * n, d, device=dev)
        ldv = (n + 3) // 4 * 4
        vt = torch.randn(nb * d, ldv, device=dev)
        khi, klo, vthi, vtlo = (torch.empty_like(t) for t in (kk, kk, vt, vt))
        _cabi.check(lib.og_split_tf32(p(kk), p(khi), p(klo), kk.numel(), st), 'og_split_tf32')
        _cabi.check(lib.og_split_tf32(p(vt), p(vthi), p(vtlo), vt.numel(), st), 'og_split_tf32')
        qq = torch.randn(nb * n, d, device=dev)

        def attn():
            _cabi.check(lib.og_attention_tc_fwd(p(qq), d, n * d, p(khi), p(klo), d, p(vthi), p(vtlo), ldv, p(o), d, n * d,
                                                nb, n, n, H, d // H, st), 'og_attention_tc_fwd')
    elif args.precision == 'fp16x3' and d // H == 64:
        def split16(x2d):
            hi = torch.empty(x2d.shape, dtype=torch.float16, device=dev)
            lo, meta = torch.empty_like(hi), torch.zeros(4, device=dev)
            _cabi.check(lib.og_weight_split_f16(p(x2d), None, x2d.shape[0], x2d.shape[1], p(hi), p(lo), p(meta), st), 'og_weight_split_f16')
            return hi, lo, meta
        kk = torch.randn(nb * n, d, device=dev)
        ldv = (n + 7) // 8 * 8
        vt = torch.randn(nb * d, ldv, device=dev)
        kh16, kl16, kmeta = split16(kk)
        vh16, vl16, vmeta = split16(vt)
        qq = torch.randn(nb * n, d, device=dev)
        qamax = torch.zeros(1, device=dev)
        _cabi.check(lib.og_amax(p(qq), qq.numel(), p(qamax), st), 'og_amax')

        def attn():
            _cabi.check(lib.og_attention_f16_fwd(p(qq), d, n * d, p(qamax), p(kh16), p(kl16), d, p(kmeta), p(vh16), p(vl16), ldv, p(vmeta),
                                                 p(o), d, n * d, None, nb, n, n, H, d // H, 0, st), 'og_attention_f16_fwd')
    else:
        def attn():
            _cabi.check(lib.og_attention_fwd(p(qkv), 3 * d, n * 3 * d, p(qkv, d), 3 * d, n * 3 * d, p(qkv, 2 * d), 3 * d,
                                             n * 3 * d, p(o), d, n * d, nb, n, n, H, d // H, prec, st), 'og_attention_fwd')
    for _ in range(3):
        attn()
    reps = 10
    ms_attn = timed(attn, reps) / reps
    attn_flops = 4.0 * n * n * d * nb
    attn_tflops = attn_flops / (ms_attn * 1e-3) / 1e12
    # secondary: the Sinkhorn kernel against the HBM roofline
    lds = (m + 3) // 4 * 4
    sbuf = torch.randn(batch, n, lds, device=dev) * 4
    sc = torch.empty(batch, n + 1, m + 1, device=dev)
    wsb = lib.og_sinkhorn_workspace_bytes(batch, n, m)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    dust = torch.ones(1, device=dev)

    def sink():
        _cabi.check(lib.og_sinkhorn_fwd(p(sbuf), lds, n * lds, p(dust), batch, n, m, iters, 1.0, p(sc), p(ws), wsb, st),
                    'og_sinkhorn_fwd')
    for _ in range(2):
        sink()
    ms_sink = timed(sink, 5) / 5
    sink_gbs = sinkhorn_bytes_per_pair(n, m, iters) * batch / (ms_sink * 1e-3) / 1e9

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    traffic = {}
    tpath = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
    if os.path.exists(tpath) and args.workload == 'C3' and batch == 16 and args.precision != 'fp32':
        traffic = json.load(open(tpath))     # ncu dram bytes per launch, captured at exactly these shapes
    fl = flops_per_pair(n, m, d, stages, s_dim)
    line = {
        'metric': METRIC, 'value': value, 'unit': 'pairs/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': max(3, args.warmup), 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None,
        'dtype': {'fp32': 'f32', 'tf32x3': 'tf32x3 (tf32 hi/lo operands, 3 products, fp32 accumulate)',
                  'fp16x3': 'fp16x3 (fp16 hi/lo operands with power-of-two tensor scales, 3 products, fp32 accumulate)'}[args.precision],
        'data': 'synthetic', 'config': bench_config(args, wl, batch),
        'e2e': {'value': e2e_value, 'unit': 'pairs/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'ms_per_step': ms_e2e / args.steps, 'api': 'MatchingCore.submit()/wait(), host buffers, 2 batches in flight',
                'blocking_forward_value': batch * world / (ms_e2e_serial / args.steps * 1e-3),
                'blocking_forward_ms_per_step': ms_e2e_serial / args.steps},
        'gpu_launches': launches,
        'verified': verified,
        'loss': ({'loss': float(loss_acc[0]), 'metric_loss': float(loss_acc[1]), 'reduced_over_ranks': world,
                  'how': 'og_gt_matches_fwd labels -> og_superglue_forward -> og_criterion_fwd per rank, NCCL all-reduce (mean) on a side stream'}
                 if with_loss else None),
        'clocks': clocks,
        'roofline': {'kernel': 'fused attention (self layer: %d sequences x %d heads, %d x %d, Dh=%d)' % (nb, H, n, n, d // H),
                     'bound': 'tensor', 'achieved': attn_tflops, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s',
                     'frac': attn_tflops / peaks['bf16_tflops'],
                     'traffic': traffic.get('attention_f16_self_32seq_2048' if (args.precision == 'fp16x3' and d // H == 64)
                                            else 'attention_tc_self_32seq_2048', {}).get('bytes') if args.workload == 'C3' else None,
                     'peak_source': peaks['source'] + ' bf16 burst',
                     'ms_per_launch': ms_attn, 'flops_per_launch': attn_flops,
                     # the kernel runs 3 MMAs per algorithmic product (fp32-grade accuracy is part of the contract): its own ceiling
                     # is bf16_peak / 6 with tf32 operands (half rate) and bf16_peak / 3 with fp16 operands
                     'frac_of_3x_ceiling': (attn_tflops / (peaks['bf16_tflops'] / (3.0 if (args.precision == 'fp16x3' and d // H == 64) else 6.0))
                                            if args.precision != 'fp32' else None)},
        'roofline_sinkhorn': {'kernel': 'sinkhorn (%d pairs, %d iterations, one launch)' % (batch, iters), 'bound': 'hbm',
                              'achieved': sink_gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                              'frac': sink_gbs / peaks['hbm_gbs'],
                              'traffic': traffic.get('sinkhorn_16pairs_2048_100it', {}).get('bytes') if args.workload == 'C3' else None,
                              'peak_source': peaks['source'],
                              'ms_per_launch': ms_sink, 'bytes_per_launch': sinkhorn_bytes_per_pair(n, m, iters) * batch},
        'flops_per_pair': fl['total'],
        'end_to_end_tensor_frac': value / world * fl['total'] / (peaks['bf16_tflops_sustained'] * 1e12),
    }
    if world == 1 and not args.no_cpu_baseline:
        r = time_oracle(args.workload, default_config(**wl['cfg']), n, m, 3)
        agg = r.get('aggregate', 0.0)
        line['cpu_baseline'] = {'value': max(r['single'], agg), 'unit': 'pairs/s',
                                'cores': r['procs'] * r['cores_per_proc'] if agg >= r['single'] else r['threads'], 'kind': _reference_kind(),
                                'single_process': r['single'], 'aggregate': agg,
                                'sample': f'single pairs of the {args.workload} shape (N={n}, M={m}), torch CPU fp32 ({"unmodified reference module, oracle/_ref" if _reference_kind() == "reference" else "oracle port"}); one process '
                                          f'pinned to NUMA node 0 ({r["node0_cpus"]} cpus, {r["threads"]} threads, best of 3 after warm-up): '
                                          f'{r["single"]:.3f} pairs/s; {r["procs"]} processes x {r["cores_per_proc"]} pinned cores side by side: '
                                          f'{agg:.3f} pairs/s aggregate; value = the larger; host: {r["cpus"]} cpus, {r["numa_nodes"]} NUMA nodes'}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
