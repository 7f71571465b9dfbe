"""Throughput of float64 flows against the same flows in float32 on the CUDA-core kernels.

    python tools/float64_throughput.py [--rows 1048576] [--train-rows 65536] [--reps 5] [--out result.json]

The headline flow (d = 64, 8 couplings, K = 16, MLP[64]; quadratic and cubic splines) is timed in one process:
  log_prob at --rows rows (no gradient: one C call per flow), and one NLL step (-log_prob.mean(), backward, Adam step)
  at --train-rows rows, each in float64 and in float32 with STRIBOR_B200_FORCE_GENERIC=1 (the CUDA-core kernels the
  float64 path runs, so the two differ only in the scalar type).
Times are CUDA-event times of a whole call, after warm-up, median of --reps.  The card's name and power limit are read in
the same process and printed with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import stribor_b200 as st  # noqa: E402


def headline(kind, dim=64):
    P = 47 if kind == 'quadratic' else 34
    masks = ('ordered_right_half', 'ordered_left_half')
    return st.NormalizingFlow(st.UnitNormal(dim), [
        st.Coupling(st.Spline(dim, 16, latent_net=st.net.MLP(dim, [64], dim * P), lower=-4., upper=4.,
                              spline_type=kind), masks[i % 2]) for i in range(8)])


def timed(fn, reps, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return sorted(ts)[len(ts) // 2]


def card():
    name = torch.cuda.get_device_name()
    try:
        power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i',
                                str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power or 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rows', type=int, default=1 << 20)
    ap.add_argument('--train-rows', type=int, default=1 << 16)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None, help='also write the results as JSON to this path')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('float64_throughput: no CUDA device; nothing is measured without one')
    name, power = card()
    os.environ['STRIBOR_B200_FORCE_GENERIC'] = '1'
    results = {'gpu': name, 'power_limit': power, 'rows': a.rows, 'train_rows': a.train_rows, 'cases': []}
    for kind in ('quadratic', 'cubic'):
        torch.manual_seed(0)
        base = headline(kind).cuda()
        for dtype in (torch.float32, torch.float64):
            flow = headline(kind).cuda().to(dtype)
            flow.load_state_dict(base.state_dict())
            y = (torch.randn(a.rows, 64, device='cuda') * 1.5).to(dtype)
            with torch.no_grad():
                lp_ms = timed(lambda: flow.log_prob(y), a.reps)
            opt = torch.optim.Adam(flow.parameters(), lr=1e-4)
            xt = y[:a.train_rows].clone()

            def step():
                opt.zero_grad(set_to_none=True)
                (-flow.log_prob(xt).mean()).backward()
                opt.step()

            step_ms = timed(step, a.reps)
            rec = {'kind': kind, 'dtype': str(dtype).replace('torch.', ''), 'log_prob_ms': round(lp_ms, 3),
                   'log_prob_rows_per_s': round(a.rows / lp_ms * 1e3), 'nll_step_ms': round(step_ms, 3),
                   'nll_step_rows_per_s': round(a.train_rows / step_ms * 1e3)}
            results['cases'].append(rec)
            print(json.dumps(rec), flush=True)
            del flow, opt, y, xt
            torch.cuda.empty_cache()
    print(json.dumps({'gpu': name, 'power_limit': power}))
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(results, f, indent=1)


if __name__ == '__main__':
    main()
