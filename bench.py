#!/usr/bin/env python
"""Headline benchmark: flow.log_prob samples/s of an 8-layer spline-coupling flow, d=64
(BASELINE.json metric / configs[2]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--kind quadratic|cubic] [--hidden 64] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...        # the CPU arm (oracle port of the reference)

One step = one log_prob pass over the global batch of 2^22 rows (sharded by rows over the N
ranks, no data-path collective: strong scaling, total work fixed as BASELINE.json words it).
`value` is timed with CUDA events with the shard already resident in HBM; `e2e` runs the same
pass from pinned HOST memory through the public API (H2D copy of the rows and D2H copy of the
log-probabilities inside the timed region).  Prints ONE JSON line on rank 0.

Weights and inputs come from fixed seeds, so two builds run with the same arguments see the same inputs;
`--dump-outputs DIR` writes what the last timed step of each timed workload returned (`dump`) to compare them.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, 'tests', 'golden')):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch

D, LAYERS, BINS = 64, 8, 16
GLOBAL_BATCH = 1 << 22
LOWER, UPPER = -4.0, 4.0
MASKS = ('ordered_right_half', 'ordered_left_half')
METRIC = 'log_prob samples/s, 8-layer spline coupling d=64'
L2_BYTES = 126 << 20


# stdout carries the ONE JSON line and nothing else: the process's fd 1 is pointed at stderr for the whole
# run (NCCL's version banner / NCCL_DEBUG output, any library print) and the result goes to the saved fd.
_RESULT_OUT = None


def _claim_stdout():
    global _RESULT_OUT
    if _RESULT_OUT is None:
        sys.stdout.flush()
        _RESULT_OUT = os.fdopen(os.dup(1), 'w')
        os.dup2(2, 1)


def emit(obj):
    out = _RESULT_OUT if _RESULT_OUT is not None else sys.stdout
    out.write(json.dumps(obj) + '\n')
    out.flush()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--kind', default='quadratic', choices=['quadratic', 'cubic'])
    ap.add_argument('--hidden', type=int, nargs='+', default=[64])
    ap.add_argument('--batch', type=int, default=GLOBAL_BATCH, help='global batch (rows)')
    ap.add_argument('--cpu-sample', type=int, default=1 << 15, help='rows of the cpu_baseline sample')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-configs', action='store_true', help='headline only: skip the cubic / affine / neural / train side configs')
    ap.add_argument('--parity-rows', type=int, default=8192, help='rows of the timed batch re-checked against the oracle')
    ap.add_argument('--generic', action='store_true', help='force the CUDA-core path (no tcgen05)')
    ap.add_argument('--micro-rows', type=int, default=1 << 18, help='train: rows per micro-batch')
    ap.add_argument('--tf32', action='store_true', help='train: let the library GEMMs of the conditioner gradients use TF32')
    ap.add_argument('--hybrid', action='store_true', help='train: conditioner through autograd around the element-wise kernels')
    ap.add_argument('--workload', default='logprob', choices=['logprob', 'cubic', 'quadratic_h256', 'affine', 'neural', 'train'],
                    help='logprob = BASELINE.json configs[2] (the headline, default); affine = configs[1]; '
                         'neural = configs[3]; train = configs[4] (side measurements, same JSON schema)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last timed step returned as DIR/<name>.npy (see dump)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    return args


def build_layers(kind, hidden):
    """Random-init conditioners with the reference's defaults (nn.Linear init, last bias 0,
    net/mlp.py:46-53), seeded on the CPU so every rank and the CPU baseline share the weights."""
    import stribor_b200 as st
    torch.manual_seed(123)
    P = 3 * BINS - 1 if kind == 'quadratic' else 2 * BINS + 2
    layers = []
    for i in range(LAYERS):
        net = st.net.MLP(D, list(hidden), D * P)
        tr = st.Spline(D, BINS, latent_net=net, lower=LOWER, upper=UPPER, spline_type=kind)
        layers.append(st.Coupling(tr, mask=MASKS[i % 2]))
    return layers


def dump(dirname, outputs, max_elems):
    """Write the outputs of the last timed step, {name: tensor}, as dirname/<name>.npy in float32 (float64 stays
    float64), rank 0's rows.  A tensor of more than `max_elems` elements is written as a fixed sample of its rows
    (first dimension): the rows a generator seeded with 0 draws first, in ascending order, the same in every run
    of the same shape.  The callers' limits keep all files of one run under 64 MB."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach()
        if t.numel() > max_elems:
            keep = max(1, max_elems // (t[0].numel() if t.dim() > 1 else 1))
            idx = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t[idx.to(t.device)]
        a = t.cpu().numpy()
        np.save(os.path.join(dirname, name + '.npy'), a if a.dtype == np.float64 else a.astype(np.float32))


def workload_name(kind, hidden, batch):
    return (f'{kind} st.Spline coupling flow d={D}, {LAYERS} layers alternating {MASKS[0]}/{MASKS[1]}, '
            f'{BINS} bins, MLP{list(hidden)} tanh, box [{LOWER:g},{UPPER:g}], log_prob, global batch {batch}')


# -------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md)
# -------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '50',
                 '-i', str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ts, line in self.samples:
            f = [v.strip() for v in line.split(',')]
            if len(f) < 6:
                continue
            try:
                clk, m = float(f[0]), float(f[1])
            except ValueError:
                continue
            mx = m
            if t0 <= ts <= t1 + 0.2:
                sm.append(clk)
                for n, v in zip(names, f[2:6]):
                    if v.lower().startswith('active'):
                        reasons.add(n)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


# -------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference, all host threads
# -------------------------------------------------------------------------------------------
def cpu_log_prob_rate(spec, kind, rows, chunk=1 << 13, repeats=1):
    from oracle import coupling_flow_oracle as O
    n_threads = len(os.sched_getaffinity(0))
    torch.set_num_threads(n_threads)
    g = torch.Generator().manual_seed(0)
    y = torch.randn(rows, D, generator=g)
    best = None
    with torch.no_grad():
        O.flow_log_prob(spec, y[:256])                       # warm-up
        for _ in range(repeats):
            t = time.perf_counter()
            for i in range(0, rows, chunk):
                O.flow_log_prob(spec, y[i:i + chunk])
            dt = time.perf_counter() - t
            best = dt if best is None else min(best, dt)
    return rows / best, n_threads, best


def cpu_model():
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                return line.split(':', 1)[1].strip()
    except Exception:
        pass
    return 'unknown'


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from stribor_b200.spec import spec_from_layers
    spec = spec_from_layers(build_layers(args.kind, args.hidden))
    rows = 1 << 13                                            # bounded sample per step
    from oracle import coupling_flow_oracle as O
    n_threads = len(os.sched_getaffinity(0))
    torch.set_num_threads(n_threads)
    y = torch.randn(rows, D, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        for _ in range(args.warmup):
            O.flow_log_prob(spec, y)
        t = time.perf_counter()
        for _ in range(args.steps):
            lp = O.flow_log_prob(spec, y)
        dt = time.perf_counter() - t
    if args.dump_outputs:
        dump(args.dump_outputs, {'log_prob': lp}, 1 << 22)
    value = rows * args.steps / dt
    sample = (f'{rows} rows per step of the same workload; oracle port of the reference (torch CPU ops, '
              f'no O(N^2) domain re-check), {n_threads} threads, {cpu_model()}')
    emit({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'samples/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic', 'config': {'workload': workload_name(args.kind, args.hidden, args.batch)},
        'cpu_baseline': {'value': value, 'unit': 'samples/s', 'cores': n_threads, 'kind': 'port',
                         'sample': sample},
        'e2e': {'value': value, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    })


# -------------------------------------------------------------------------------------------
# the other BASELINE.json configs: cubic (configs[2], second half), affine (configs[1]), neural (configs[3]),
# train (configs[4]).  The default command line reports them under the `configs` key of the ONE JSON line,
# after the headline; `--workload X` prints X alone.
# -------------------------------------------------------------------------------------------
def _peaks():
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        pk = json.load(open(peaks_path))
        return (float(pk['hbm_gbs']), float(pk.get('bf16_tflops_sustained', pk.get('bf16_tflops', 1394.6))),
                'measured (MEASURED_PEAKS.json: hbm_gbs, bf16_tflops_sustained)')
    return 6650.0, 1400.0, 'fallback (B200_PROFILING.md)'


def _profile_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per row of the dominant kernel, from the committed
    `ncu --set full` summaries (profiles/r02_traffic.json, else r01), or None"""
    for f in ('r02_traffic.json', 'r01_traffic.json'):
        path = os.path.join(ROOT, 'profiles', f)
        if os.path.exists(path):
            tj = json.load(open(path))
            if key in tj:
                return tj[key]
    return None


def _timed(step, steps, warmup, dev, world):
    """W warm-up steps, K timed steps between barriers; CUDA events on the launching stream, max over ranks.
    -> (ms per step, library launches inside the timed region, what the last step returned)"""
    import torch.distributed as dist
    from stribor_b200 import _ops

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(warmup):
        step()
    barrier()
    n0 = _ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = step()
    e1.record()
    barrier()
    tm = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    return tm.item() / steps, int(_ops.launch_count() - n0), out


def _cpu_rate(fn, units, min_seconds=0.0):
    """`fn()` once for warm-up on a small slice is the caller's business; here: one timed call"""
    n_threads = len(os.sched_getaffinity(0))
    torch.set_num_threads(n_threads)
    t = time.perf_counter()
    fn()
    dt = time.perf_counter() - t
    return units / dt, n_threads, dt


def _parity_block(got, w32, w64, what):
    """SURVEY 8c's rule on sampled rows of the timed batch: inside rtol = atol = 1e-5 of the fp32 oracle, or no further
    from the fp64 oracle than the fp32 oracle itself is (+ the tolerance)."""
    got, w32, w64 = got.double().reshape(-1), w32.double().reshape(-1), w64.double().reshape(-1)
    tol = 1e-5 + 1e-5 * w64.abs()
    c1 = (got - w32).abs() <= tol
    c2 = (got - w64).abs() <= (w32 - w64).abs() + tol
    return {'values': int(got.numel()), 'of': what, 'rtol': 1e-5, 'atol': 1e-5,
            'frac_outside': float(1.0 - (c1 | c2).double().mean()),
            'frac_needing_fp64_arbitration': float(((~c1) & c2).double().mean()),
            'max_abs': float((got - w64).abs().max()), 'oracle_fp32_max_abs': float((w32 - w64).abs().max()),
            'rule': '|new-ref32| <= atol+rtol|ref| or |new-ref64| <= |ref32-ref64| + atol+rtol|ref| (SURVEY 8c)'}


def side_config(workload, args, dev, rank, world, want_cpu):
    """One side configuration -> its result dict (same fields as the headline: value / e2e / roofline /
    cpu_baseline).  Rows are sharded over the ranks exactly like the headline."""
    import stribor_b200 as st
    from stribor_b200.host import HostPipeline
    from stribor_b200.parallel import DataParallelNLL, shard_rows
    from stribor_b200.spec import spec_from_layers
    from oracle import coupling_flow_oracle as O          # cpu_baseline leg only (rank 0, N = 1)

    hbm_peak, tf_peak, peak_src = _peaks()
    steps, warmup = args.steps, args.warmup
    torch.manual_seed(123)
    res = {'steps': steps, 'warmup': warmup, 'n_gpus': world, 'higher_is_better': True, 'scaling': 'strong',
           'dtype': 'f32', 'data': 'synthetic'}
    cpu = None
    if workload in ('cubic', 'quadratic_h256'):
        d, rows_g = D, args.batch if workload == 'cubic' else args.batch // 4
        kind_w, hid_w = ('cubic', [64]) if workload == 'cubic' else ('quadratic', [256, 256])
        layers = build_layers(kind_w, hid_w)
        flow = st.NormalizingFlow(st.UnitNormal(d), layers).to(dev).requires_grad_(False)
        a, b = shard_rows(rows_g, rank, world)
        y = torch.randn(b - a, d, device=dev, generator=torch.Generator(dev).manual_seed(rank))
        name = workload_name(kind_w, hid_w, rows_g)

        def step():
            with torch.no_grad():
                return flow.log_prob(y)
        unit, per_step = 'samples/s', rows_g
        ins, n_out = [y], 1
        out_names = ('log_prob',)
        pipe_fn = lambda yy: flow.log_prob(yy)
        if workload == 'cubic':
            bytes_unit, flops_unit, bound = LAYERS * (8 * d + 8), 2 * (32 * 64 + 64 * 32 * 34) * LAYERS, 'hbm'
            traffic_key = 'cubic_dram_bytes_per_row_chain'
        else:        # SURVEY 8d's secondary configs[2] shape: 917 504 flop per row and layer
            bytes_unit, flops_unit, bound = LAYERS * (8 * d + 8), 2 * (32 * 256 + 256 * 256 + 256 * 32 * 47) * LAYERS, 'tensor'
            traffic_key = None
        if want_cpu:
            spec = spec_from_layers([l.cpu() for l in build_layers(kind_w, hid_w)])
            n = 1 << 13
            yc = torch.randn(n, d, generator=torch.Generator().manual_seed(0))
            with torch.no_grad():
                O.flow_log_prob(spec, yc[:256])
                cpu = _cpu_rate(lambda: O.flow_log_prob(spec, yc), n) + (f'{n} rows of the same workload, one call',)
    elif workload == 'affine':
        d, rows_g = 64, 1 << 20
        layers = [st.Coupling(st.Affine(d, latent_net=st.net.MLP(d, [256, 256], 2 * d)), mask=MASKS[i % 2])
                  for i in range(LAYERS)]
        spec = spec_from_layers(layers) if want_cpu else None
        flow = st.NormalizingFlow(st.UnitNormal(d), layers).to(dev).requires_grad_(False)
        name = f'affine coupling flow d=64, 8 layers alternating masks, MLP[256,256] tanh, log_prob + inverse, global batch {rows_g}'
        a, b = shard_rows(rows_g, rank, world)
        y = torch.randn(b - a, d, device=dev, generator=torch.Generator(dev).manual_seed(rank))

        def step():
            with torch.no_grad():
                return flow.log_prob(y), flow.inverse(y)
        unit, per_step = 'samples/s (log_prob + inverse per sample)', rows_g
        ins, n_out = [y], 2
        out_names = ('log_prob', 'inverse')
        pipe_fn = lambda yy: (flow.log_prob(yy), flow.inverse(yy))
        bytes_unit = LAYERS * (8 * d + 8) + LAYERS * 8 * d
        flops_unit, bound = 2 * LAYERS * 2 * (32 * 256 + 256 * 256 + 256 * 64), 'tensor'
        traffic_key = None
        if want_cpu:
            n = 1 << 15
            yc = torch.randn(n, d, generator=torch.Generator().manual_seed(0))
            with torch.no_grad():
                O.flow_log_prob(spec, yc[:256])
                cpu = _cpu_rate(lambda: (O.flow_log_prob(spec, yc), O.flow_inverse(spec, yc)), n) + \
                    (f'{n} rows of the same workload (log_prob + inverse), one call each',)
    elif workload == 'neural':
        d, B, T, nl = 16, 65536, 64, 4
        layers = [st.ContinuousAffineCoupling(st.net.MLP(d + 1, [64], 2 * d), st.net.TimeLinear(2 * d),
                                              ('ordered_0', 'ordered_1')[i % 2]) for i in range(nl)]
        spec = spec_from_layers(layers) if want_cpu else None
        flow = st.NeuralFlow(layers).to(dev).requires_grad_(False)
        name = f'NeuralFlow 4x ContinuousAffineCoupling dim 16, MLP[17->64->32] tanh, TimeLinear(32), x [{B},{T},{d}] with per-step t, forward'
        a, b = shard_rows(B, rank, world)
        g = torch.Generator(dev).manual_seed(rank)
        x = torch.randn(b - a, T, d, device=dev, generator=g)
        t = torch.rand(b - a, T, 1, device=dev, generator=g)

        def step():
            with torch.no_grad():
                return flow(x, t=t)
        unit, per_step = 'rows/s', B * T
        ins, n_out = [x, t], 1
        out_names = ('y',)
        pipe_fn = lambda xx, tt: flow(xx, t=tt)
        bytes_unit, flops_unit, bound = nl * (2 * 4 * d + 4), nl * 2 * (9 * 64 + 64 * 16), 'hbm'
        traffic_key = 'neural_dram_bytes_per_row'
        if want_cpu:
            n = 1 << 12
            gc = torch.Generator().manual_seed(0)
            xc, tc = torch.randn(n, T, d, generator=gc), torch.rand(n, T, 1, generator=gc)
            with torch.no_grad():
                O.neural_flow_forward(spec, xc[:8], tc[:8])
                cpu = _cpu_rate(lambda: O.neural_flow_forward(spec, xc, tc), n * T) + \
                    (f'x [{n},{T},{d}] of the same workload, one call',)
    else:
        d, rows_g = 128, args.batch
        P = 3 * BINS - 1
        layers = [st.Coupling(st.Spline(d, BINS, latent_net=st.net.MLP(d, list(args.hidden), d * P), lower=LOWER,
                                        upper=UPPER, spline_type='quadratic'), mask=MASKS[i % 2])
                  for i in range(LAYERS)]
        spec = spec_from_layers(layers) if want_cpu else None
        flow = st.NormalizingFlow(st.UnitNormal(d), layers).to(dev)
        name = (f'NLL training step (fwd+bwd, gradients and loss all-reduced over NCCL) quadratic spline coupling d=128, '
                f'8 layers, 16 bins, MLP{list(args.hidden)} tanh, global batch {rows_g}')
        a, b = shard_rows(rows_g, rank, world)
        y = torch.randn(b - a, d, device=dev, generator=torch.Generator(dev).manual_seed(rank))
        if args.tf32:
            torch.backends.cuda.matmul.allow_tf32 = True
        if args.hybrid:
            os.environ['STRIBOR_B200_TRAIN_HYBRID'] = '1'
        name += (f', micro-batches of {args.micro_rows} rows' + (', hybrid path' if args.hybrid else ', fused backward kernel'))
        dp = DataParallelNLL(flow, micro_rows=args.micro_rows)

        def step():
            return dp.step(y, rows_g)
        unit, per_step = 'samples/s', rows_g
        ins, n_out = [y], 0
        out_names = ('loss',)               # and the gradients, all-reduced, as one flat 'grad'
        pipe_fn = None
        bytes_unit = LAYERS * (8 * d + 8) + LAYERS * 12 * d
        flops_unit, bound = 3 * LAYERS * 2 * (64 * 64 + 64 * 64 * P), 'tensor'
        traffic_key = None
        if want_cpu:
            n = 1 << 11
            yc = torch.randn(n, d, generator=torch.Generator().manual_seed(0))
            leaves = []
            for layer in spec:
                net = layer['transform']['net']
                for w, bb in zip(net['weights'], net['biases']):
                    leaves += [w.requires_grad_(True), bb.requires_grad_(True)]

            def cpu_step():
                (-O.flow_log_prob(spec, yc).mean()).backward()
            cpu_step()
            cpu = _cpu_rate(cpu_step, n) + (f'{n} rows, one fwd+bwd of the same flow through torch autograd on the oracle port',)

    ms_step, launches, last = _timed(step, steps, warmup, dev, world)
    if args.dump_outputs and rank == 0:
        outs = dict(zip(out_names, last if isinstance(last, (tuple, list)) else (last,)))
        if workload == 'train':
            outs['grad'] = torch.cat([p.grad.reshape(-1) for p in flow.parameters()])
        dump(args.dump_outputs, {f'{workload}.{k}': v for k, v in outs.items()}, 1 << 20)
    value = per_step / (ms_step * 1e-3)
    rows_local = ins[0].shape[0] * (ins[0].shape[1] if workload == 'neural' else 1)
    res.update({'metric': f'{workload} throughput', 'value': value, 'unit': unit, 'ms_per_step': ms_step,
                'config': {'workload': name, 'l2_policy': 'inputs larger than L2' if ins[0].numel() * 4 > L2_BYTES
                           else 'inputs + outputs of one step exceed L2 together'},
                'gpu_launches': launches})
    # roofline of the config's dominant kernel family: algorithmic bytes (SURVEY 8d) or masked-minimum flops
    # per unit x the units this rank processes per step / measured step time (the step is that kernel family
    # back to back; nothing else runs in the timed region)
    if bound == 'hbm':
        ach = rows_local * bytes_unit / (ms_step * 1e-3) / 1e9
        tr = _profile_traffic(traffic_key) if traffic_key else None
        res['roofline'] = {'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach / hbm_peak,
                           'traffic': None if tr is None else tr * rows_local / max(launches / steps, 1),
                           'peak_source': peak_src, 'bytes_per_unit': bytes_unit,
                           'binding': 'tensor pipe + spline epilogue (SURVEY 8d)' if workload == 'cubic' else 'hbm'}
        res['roofline_tensor'] = {'bound': 'tensor', 'achieved': rows_local * flops_unit / (ms_step * 1e-3) / 1e12,
                                  'peak': tf_peak, 'unit': 'TFLOP/s',
                                  'frac': rows_local * flops_unit / (ms_step * 1e-3) / 1e12 / tf_peak,
                                  'note': 'masked-minimum fp32-equivalent conditioner flops over the measured bf16 dense peak'}
    else:
        ach = rows_local * flops_unit / (ms_step * 1e-3) / 1e12
        res['roofline'] = {'bound': 'tensor', 'achieved': ach, 'peak': tf_peak, 'unit': 'TFLOP/s', 'frac': ach / tf_peak,
                           'traffic': None, 'peak_source': peak_src, 'flops_per_unit': flops_unit,
                           'note': 'masked-minimum fp32-equivalent conditioner flops (SURVEY 8d) over the measured bf16 '
                                   'dense peak; the kernels issue kind::f16 tcgen05.mma in 3 split passes, i.e. ~3x these flops'}
        res['roofline_hbm'] = {'bound': 'hbm', 'achieved': rows_local * bytes_unit / (ms_step * 1e-3) / 1e9,
                               'peak': hbm_peak, 'unit': 'GB/s',
                               'frac': rows_local * bytes_unit / (ms_step * 1e-3) / 1e9 / hbm_peak}
    # end to end: pinned host buffers -> H2D -> the public call -> D2H, inside the timed region
    if pipe_fn is not None and not args.no_e2e:
        chunk = max(1 << 12, ins[0].shape[0] // 4)
        pipe = HostPipeline(flow, d, dev, chunk_rows=chunk)
        ins_h = [torch.empty(t_.shape, pin_memory=True).copy_(t_) for t_ in ins]
        with torch.no_grad():
            sample = pipe_fn(*[t_[:2] for t_ in ins])
        sample = sample if isinstance(sample, (tuple, list)) else (sample,)
        outs_h = [torch.empty((ins[0].shape[0],) + tuple(o.shape[1:]), pin_memory=True) for o in sample]
        k = 3
        ms_e = _timed(lambda: pipe.map(pipe_fn, ins_h, outs_h), k, 2, dev, world)[0]
        res['e2e'] = {'value': per_step / (ms_e * 1e-3), 'unit': unit,
                      'h2d_bytes_per_step': sum(t_.numel() * 4 for t_ in ins_h) * world,
                      'd2h_bytes_per_step': sum(o.numel() * 4 for o in outs_h) * world,
                      'how': f'pinned host tensors -> H2D -> public call -> D2H, chunks of {chunk} rows on two streams'}
    elif workload == 'train':
        # the training step's host traffic: the batch arrives from pinned host memory every step, the scalar loss
        # goes back (what a data loader feeds); gradients stay on the device for the optimizer
        y_h = torch.empty(y.shape, pin_memory=True).copy_(y)
        ybuf = torch.empty_like(y)

        def e2e_step():
            ybuf.copy_(y_h, non_blocking=True)
            return float(dp.step(ybuf, rows_g))
        ms_e = _timed(e2e_step, 2, 1, dev, world)[0]
        res['e2e'] = {'value': per_step / (ms_e * 1e-3), 'unit': unit, 'h2d_bytes_per_step': y_h.numel() * 4 * world,
                      'd2h_bytes_per_step': 4 * world, 'how': 'pinned host batch -> H2D -> DataParallelNLL.step -> loss.item()'}
        res['allreduce_bytes_per_step'] = int(dp.last_allreduce_bytes)
    # parity of the timed inputs: sampled rows re-evaluated by the oracle in fp32 and fp64 (rank 0, with the CPU legs)
    if want_cpu and workload != 'train' and args.parity_rows > 0:
        n = min(2048, args.parity_rows, ins[0].shape[0])
        idx = torch.randperm(ins[0].shape[0], generator=torch.Generator().manual_seed(7))[:n].sort().values.to(dev)
        sub = [t_[idx] for t_ in ins]
        with torch.no_grad():
            got = pipe_fn(*sub)
        got = got if isinstance(got, (tuple, list)) else (got,)
        spec_p = spec_from_layers([l.cpu() for l in build_layers(kind_w, hid_w)]) if workload in ('cubic', 'quadratic_h256') else spec
        s64 = O.spec_to(spec_p, torch.float64)
        subc = [t_.cpu() for t_ in sub]
        torch.set_num_threads(len(os.sched_getaffinity(0)))
        with torch.no_grad():
            if workload == 'neural':
                w32 = (O.neural_flow_forward(spec_p, subc[0], subc[1]),)
                w64 = (O.neural_flow_forward(s64, subc[0].double(), subc[1].double()),)
            elif workload == 'affine':
                w32 = (O.flow_log_prob(spec_p, subc[0]), O.flow_inverse(spec_p, subc[0]))
                w64 = (O.flow_log_prob(s64, subc[0].double()), O.flow_inverse(s64, subc[0].double()))
            else:
                w32 = (O.flow_log_prob(spec_p, subc[0]),)
                w64 = (O.flow_log_prob(s64, subc[0].double()),)
        blocks = [_parity_block(g.cpu(), a, b, f'{n} rows of the timed batch, fixed seed') for g, a, b in zip(got, w32, w64)]
        res['parity'] = blocks[0] if len(blocks) == 1 else {'log_prob': blocks[0], 'inverse': blocks[1]}
    if cpu is not None:
        v, cores, secs, what = cpu
        res['cpu_baseline'] = {'value': v, 'unit': unit, 'cores': cores, 'kind': 'port',
                               'sample': f'{what} ({secs:.1f} s); oracle port of the reference on torch CPU ops, '
                                         f'{cores} threads, {cpu_model()}'}
    return res


def run_side(args):
    from stribor_b200.parallel import init_from_env
    rank, world, local = init_from_env('nccl')
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    res = side_config(args.workload, args, dev, rank, world, want_cpu=(world == 1 and not args.no_cpu_baseline))
    if rank == 0:
        res.setdefault('vs_baseline', None)
        emit(res)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


# -------------------------------------------------------------------------------------------
# GPU arm
# -------------------------------------------------------------------------------------------
def main():
    args = parse()
    _claim_stdout()
    if args.impl == 'reference':
        run_reference(args)
        return
    if args.workload != 'logprob':
        run_side(args)
        return

    import torch.distributed as dist
    import stribor_b200 as st
    from stribor_b200 import _ops
    from stribor_b200.host import HostPipeline

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit(f'--gpus {args.gpus} needs torchrun with {args.gpus} ranks')
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    from stribor_b200.parallel import bind_to_gpu_numa
    numa = bind_to_gpu_numa(local) if world > 1 else {'bound': False, 'why': 'single process'}
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    layers = build_layers(args.kind, args.hidden)
    flow = st.NormalizingFlow(st.UnitNormal(D), layers).to(dev)
    if args.generic:
        os.environ['STRIBOR_B200_FORCE_GENERIC'] = '1'
    for p in flow.parameters():
        p.requires_grad_(False)

    rows = args.batch // world
    torch.manual_seed(rank)
    y = torch.randn(rows, D, device=dev)                      # 2^22 x 64 fp32 = 1 GiB  (> 126 MB L2)

    def step():
        with torch.no_grad():
            return flow.log_prob(y)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks are sampled from the start of the warm-up (identical load) to the end of the timed
    # region, so that short timed regions (strong scaling at 8 GPUs: ~20 ms) still get samples
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.25)
    t_load0 = time.perf_counter()
    for _ in range(args.warmup):
        step()
    barrier()
    n0 = _ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        lp = step()
    e1.record()
    barrier()
    t1 = time.perf_counter()
    launches = _ops.launch_count() - n0
    ms = e0.elapsed_time(e1)
    if t1 - t_load0 < 0.35:                                # keep the GPU under the same load until a sample lands
        while time.perf_counter() - t_load0 < 0.35:
            step()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
    clocks = sampler.stop(t_load0, t1)
    clocks['window'] = 'warm-up + timed steps (same workload)'
    assert torch.isfinite(lp).all().item(), 'non-finite log_prob'
    if args.dump_outputs and rank == 0:
        dump(args.dump_outputs, {'log_prob': lp}, 1 << 22)
    tmax = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_step = tmax.item() / args.steps
    value = args.batch / (ms_step * 1e-3)

    # ---- end to end: pinned host rows -> device -> log_prob -> host -------------------------
    e2e = None
    if not args.no_e2e:
        pipe = HostPipeline(flow, D, dev, chunk_rows=max(1 << 16, min(1 << 18, rows // 6)), n_streams=3)
        y_host = torch.empty(rows, D, pin_memory=True)
        y_host.copy_(y)
        lp_host = torch.empty(rows, 1, pin_memory=True)
        for _ in range(2):
            pipe.log_prob(y_host, lp_host)
        barrier()
        k = max(2, min(args.steps, 5))
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(k):
            pipe.log_prob(y_host, lp_host)
        s1.record()
        barrier()
        te = torch.tensor([s0.elapsed_time(s1)], device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        assert torch.allclose(lp_host, lp.cpu(), rtol=0, atol=0), 'e2e result differs from device result'
        e2e = {'value': args.batch / (te.item() / k * 1e-3), 'unit': 'samples/s',
               'h2d_bytes_per_step': rows * D * 4 * world, 'd2h_bytes_per_step': rows * 4 * world,
               'how': f'pinned host rows -> H2D -> flow.log_prob -> D2H, chunks of {pipe.chunk_rows} rows '
                      f'on {len(pipe.streams)} streams', 'numa': numa}

    # ---- parity of the TIMED batch: sampled rows re-evaluated by the oracle (fp32 and fp64) -------------
    parity = None
    if rank == 0 and args.parity_rows > 0 and not args.no_cpu_baseline:
        from oracle import coupling_flow_oracle as O          # the checker, after the timed region
        from stribor_b200.spec import spec_from_layers
        n = min(args.parity_rows, rows)
        idx = torch.randperm(rows, generator=torch.Generator().manual_seed(7))[:n].sort().values
        ys = y[idx.to(dev)].cpu()
        got = lp[idx.to(dev)].cpu().double().view(-1)
        spec = spec_from_layers([l.cpu() for l in build_layers(args.kind, args.hidden)])
        torch.set_num_threads(len(os.sched_getaffinity(0)))
        with torch.no_grad():
            w32 = torch.cat([O.flow_log_prob(spec, ys[i:i + 2048]) for i in range(0, n, 2048)]).double().view(-1)
            s64 = O.spec_to(spec, torch.float64)
            w64 = torch.cat([O.flow_log_prob(s64, ys[i:i + 2048].double()) for i in range(0, n, 2048)]).view(-1)
        tol = 1e-5 + 1e-5 * w64.abs()
        c1 = (got - w32).abs() <= tol
        c2 = (got - w64).abs() <= (w32 - w64).abs() + tol
        parity = {'rows': int(n), 'of': 'the timed batch, rows drawn with a fixed seed', 'rtol': 1e-5, 'atol': 1e-5,
                  'frac_outside': float(1.0 - (c1 | c2).double().mean()),
                  'frac_needing_fp64_arbitration': float(((~c1) & c2).double().mean()),
                  'max_abs': float((got - w64).abs().max()), 'oracle_fp32_max_abs': float((w32 - w64).abs().max()),
                  'rule': '|new-ref32| <= atol+rtol|ref| or |new-ref64| <= |ref32-ref64| + atol+rtol|ref| (SURVEY 8c)'}

    # ---- roofline of the dominant kernel (one fused layer launch) ---------------------------
    hbm_peak, tf_peak, peak_src = _peaks()
    launch_ms = ms / max(launches, 1)                         # rank-local average launch duration
    # layer applications one launch performs: 1 (a launch per layer) or all L (whole flow in one launch,
    # the tile stays in shared memory between layers -- DRAM traffic is then ~L times below the algorithmic
    # figure, which by SURVEY 8d stays L * (8d + 8) B per sample)
    layers_per_launch = LAYERS * args.steps / max(launches, 1)
    bytes_per_launch = rows * (8 * D + 8) * layers_per_launch  # per layer: read y + write x + read/write ldj
    achieved = bytes_per_launch / (launch_ms * 1e-3) / 1e9
    P = 3 * BINS - 1 if args.kind == 'quadratic' else 2 * BINS + 2
    h = [D // 2] + list(args.hidden)
    flops_row = 2 * (sum(a * b for a, b in zip(h[:-1], h[1:])) + h[-1] * (D // 2) * P)
    tflops = rows * flops_row * layers_per_launch / (launch_ms * 1e-3) / 1e12
    traffic = None
    if args.kind == 'quadratic' and not args.generic:             # dram__bytes_{read,write}.sum from ncu --set full
        per_row = _profile_traffic('dram_bytes_per_row_chain' if layers_per_launch > 1 else 'dram_bytes_per_row')
        traffic = None if per_row is None else per_row * rows
    roofline = {'bound': 'hbm', 'achieved': achieved, 'peak': hbm_peak, 'unit': 'GB/s',
                'frac': achieved / hbm_peak, 'traffic': traffic, 'peak_source': peak_src,
                'kernel': 'fused coupling layer' + (f', {layers_per_launch:g} layers per launch (tile resident in shared memory)'
                                                    if layers_per_launch > 1 else ' (one launch per layer)'),
                'layers_per_launch': layers_per_launch,
                'bytes_per_launch': bytes_per_launch, 'launch_ms': launch_ms,
                'note': 'BASELINE metric asks for % of HBM peak on L*(8d+8) B/sample; the kernel is '
                        'bound by the conditioner contraction + spline epilogue, see tensor figure'}
    # executed tensor work: GEMM1 as 8 bf16 partial products of [rows x 32] x [32 x 64], GEMM2 as 3 fp16 passes
    # over 48 (padded from 47 / 34) columns per transformed dim
    exec_flops_row = 2 * (8 * 32 * 64 + 3 * 64 * (D // 2) * 48) if list(args.hidden) == [64] else None
    roofline_tensor = {'bound': 'tensor', 'achieved': tflops, 'peak': tf_peak, 'unit': 'TFLOP/s',
                       'frac': tflops / tf_peak,
                       'note': 'numerator: masked-minimum fp32-EQUIVALENT conditioner flops (SURVEY 8d); denominator: '
                               'measured bf16 dense peak, while the kernel issues kind::f16 tcgen05.mma (same rate) in '
                               'split passes -- see executed_*'}
    if exec_flops_row is not None and not args.generic:
        ex = rows * exec_flops_row * layers_per_launch / (launch_ms * 1e-3) / 1e12
        roofline_tensor.update({'executed_tflops': ex, 'executed_frac': ex / tf_peak,
                                'executed_over_useful': exec_flops_row / flops_row})

    out = {
        'metric': METRIC, 'value': value, 'unit': 'samples/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'strong',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload_name(args.kind, args.hidden, args.batch),
                   'rows_per_gpu': rows, 'l2_policy': 'inputs larger than L2 (1 GiB of rows per pass)',
                   'path': 'generic' if args.generic else 'auto'},
        'clocks': clocks, 'e2e': e2e, 'gpu_launches': int(launches),
        'roofline': roofline, 'roofline_tensor': roofline_tensor, 'parity': parity,
    }

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from stribor_b200.spec import spec_from_layers
        spec = spec_from_layers([l.cpu() for l in build_layers(args.kind, args.hidden)])
        v, cores, secs = cpu_log_prob_rate(spec, args.kind, args.cpu_sample)
        out['cpu_baseline'] = {
            'value': v, 'unit': 'samples/s', 'cores': cores, 'kind': 'port',
            'sample': f'{args.cpu_sample} rows of the same workload in chunks of 8192 ({secs:.1f} s); oracle '
                      f'port of the reference on torch CPU ops, {cores} threads, {cpu_model()}; the '
                      'unmodified reference has an O(N^2) domain re-check on the quadratic path '
                      '(57 samples/s at 256-row chunks, BASELINE.md) that the port omits'}
    # ---- the other BASELINE.json configs, each with its own roofline / cpu_baseline / e2e ----------------
    if not args.no_configs and args.kind == 'quadratic' and list(args.hidden) == [64] and not args.generic \
            and args.batch == GLOBAL_BATCH:
        del y, lp
        if e2e is not None:
            del pipe, y_host, lp_host
        torch.cuda.empty_cache()
        cfgs = {}
        for w in ('cubic', 'quadratic_h256', 'affine', 'neural', 'train'):
            try:
                cfgs[w] = side_config(w, args, dev, rank, world, want_cpu=(world == 1 and not args.no_cpu_baseline))
            except Exception as e:                             # a side config must never cost the headline line
                cfgs[w] = {'error': f'{type(e).__name__}: {e}'}
            torch.cuda.empty_cache()
        out['configs'] = cfgs
    if rank == 0:
        emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
