"""HBM throughput of the functional spline API's kernels, with the reference defaults and with custom options.

    python tools/spline_functional_bw.py [--rows 1048576] [--dim 64] [--bins 16] [--iters 20] [--out FILE]

Times forward, inverse and backward of unconstrained_rational_quadratic_spline and unconstrained_cubic_spline on
per-row parameters (the row_out kernels of generic_layer.cu and backward.cu), each through the C ABI on buffers
allocated once, so the time is the kernel's.  Reports the algorithmic bytes over the median kernel time:
  forward / inverse  read x and the parameters, write y and the per-dimension log-derivative;
  backward           read x, the parameters, g_y and g_ld, write g_x and the parameter gradient.
The peak it is compared with is measured in the same run: a device-to-device copy of 4 GiB.  The working set of
every case is several GB, far beyond the 126 MB L2, so each pass streams from HBM.  Needs a GPU.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from stribor_b200 import _lib, _ops  # noqa: E402


def _median_ms(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    t = sorted(a.elapsed_time(b) for a, b in ev)
    return t[len(t) // 2]


def _hbm_peak_gbs(iters):
    n = 1 << 30                                   # 4 GiB of float32
    src = torch.empty(n, device='cuda').fill_(1.0)
    dst = torch.empty_like(src)
    ms = _median_ms(lambda: dst.copy_(src), iters)
    del src, dst
    return 2 * 4 * n / ms / 1e6


def _gpu_label():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return name, (q[torch.cuda.current_device()] if q else 'unknown')
    except (OSError, subprocess.SubprocessError):
        return name, 'unknown'


def _case(kind, K, opts, rows, dim, iters):
    """opts: None (reference defaults) or the 7 stb_spline_opts values of fmeta."""
    free = opts is not None and kind == _lib.RQS and opts[4]
    P = (3 * K + 1 if free else 3 * K - 1) if kind == _lib.RQS else 2 * K + 2
    g = torch.Generator(device='cuda').manual_seed(0)
    x = torch.rand(rows, dim, device='cuda', generator=g) * 5.0 - 2.5      # ~20 % of the elements in the tails
    prm = torch.randn(rows, dim * P, device='cuda', generator=g)
    y, ld = torch.empty_like(x), torch.empty_like(x)
    g_y, g_ld = torch.randn_like(x), torch.randn_like(x)
    g_x, g_prm = torch.empty_like(x), torch.empty_like(prm)
    meta = [kind, dim, 0, 0, 0, K, 1, 0, 0, 0, 0, 1, 0, 1]
    fmeta = [-2.0, 2.0] * 3 + (list(opts) if opts is not None else [])
    L = _ops.make_struct(meta, fmeta, None, [prm], None)
    G = _lib.StbLayerGrads()
    G.g_row_out = g_prm.data_ptr()
    lib = _lib.lib()
    s = torch.cuda.current_stream().cuda_stream

    def apply(direction):
        _lib.check(lib.stb_layer_apply_diag(C.byref(L), direction, x.data_ptr(), None, None, y.data_ptr(),
                                            ld.data_ptr(), rows, s))

    def backward():
        _lib.check(lib.stb_layer_backward_diag(C.byref(L), _lib.FORWARD, x.data_ptr(), g_y.data_ptr(), g_ld.data_ptr(),
                                               g_x.data_ptr(), C.byref(G), rows, s))

    e = 4 * rows * dim                            # bytes of one [rows, dim] float32 tensor
    out = {}
    for op, fn, nbytes in (('forward', lambda: apply(_lib.FORWARD), e * (1 + P + 2)),
                           ('inverse', lambda: apply(_lib.INVERSE), e * (1 + P + 2)),
                           ('backward', backward, e * (3 + P + 1 + P))):
        ms = _median_ms(fn, iters)
        out[op] = dict(ms=ms, gb=nbytes / 1e9, gbs=nbytes / ms / 1e6)
    return P, out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--rows', type=int, default=1 << 20)
    ap.add_argument('--dim', type=int, default=64)
    ap.add_argument('--bins', type=int, default=16)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--out', default=None, help='also write the results as JSON here')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('spline_functional_bw.py needs a CUDA device')
    K = a.bins
    cases = [
        ('rqs', _lib.RQS, 'defaults', None),
        ('rqs', _lib.RQS, 'min 1e-2 / 1e-2 / 1e-2', (1., 1e-2, 1e-2, 1e-2, 0., 0., 0.)),
        ('rqs', _lib.RQS, 'min 1e-2 / 1e-2 / 1e-2, K+1 derivatives', (1., 1e-2, 1e-2, 1e-2, 1., 0., 0.)),
        ('cubic', _lib.CUBIC, 'defaults', None),
        ('cubic', _lib.CUBIC, 'min 2e-2 / 2e-2, eps 1e-4, threshold 1e-2', (1., 2e-2, 2e-2, 0., 0., 1e-4, 1e-2)),
    ]
    name, power = _gpu_label()
    peak = _hbm_peak_gbs(a.iters)
    print(f'{name}, power limit / max SM clock: {power}')
    print(f'measured HBM peak (device-to-device copy, 4 GiB): {peak:.0f} GB/s')
    print(f'rows {a.rows}, dim {a.dim}, K {K}; median of {a.iters} launches')
    rows_out = []
    for spline, kind, label, opts in cases:
        P, res = _case(kind, K, opts, a.rows, a.dim, a.iters)
        for op, r in res.items():
            r.update(spline=spline, options=label, op=op, params_per_dim=P, share_of_peak=r['gbs'] / peak)
            rows_out.append(r)
            print(f'{spline:5s} {op:8s} {label:42s} {r["ms"]:8.3f} ms  {r["gb"]:6.2f} GB  {r["gbs"]:6.0f} GB/s  '
                  f'{100 * r["share_of_peak"]:5.1f} % of measured peak')
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(dict(gpu=name, power_limit_and_max_sm_clock=power, hbm_peak_gbs=peak, rows=a.rows, dim=a.dim,
                           bins=K, results=rows_out), f, indent=1)


if __name__ == '__main__':
    main()
