"""Record the reference's own bin indices layer by layer -> tests/golden/reference_bins.npz.

Run in the build container only (the reference does not travel to the GPU box):

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_bins.py

For every case with a spline layer (``cases.spline_cases()``) the UNMODIFIED reference layers are applied one
after the other in fp32.  ``stribor.util.searchsorted`` (util/search_sorted.py:3-5) is spied on while a spline
layer runs, and its flat result -- the reference gathers the in-box elements into a 1-D vector
(rational_quadratic_spline.py:161-164, cubic_spline.py:55-67) -- is scattered back to ``[rows, dim]`` with -1
for out-of-box elements and for the pass-through dims of a coupling (the reference transforms those too and
discards the result; the kernels never touch them).  Per spline layer ``i`` the recording holds

    x        layer input                        fwd.bins   search on cumwidths at x
    y        reference forward output           inv.bins   search on cumheights at y
    xr       reference inverse of y             inv.fbins  forward re-search at xr (couplings:
                                                           flow.py:42-47 -> coupling.py:84-95)

and ``stored_form`` writes it compactly (``tests/test_bins_golden.py:recorded_layers`` reads it back):

    case|L{i}|x        only when it is neither the case input nor the previous spline layer's y
    case|L{i}|y^x      bits of y XOR bits of x (int32; exact, and zero on the pass-through dims)
    case|L{i}|xr^x     bits of xr XOR bits of x (int32; near zero: xr is x up to the round trip)
    case|L{i}|fwd.bins, inv.bins, inv.fbins
    case|rows          the larger BIN_CASES keep a fixed half of their rows, these (sorted) ones
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, '_stubs'))
sys.path.insert(0, os.environ.get('STRIBOR_REFERENCE', '/root/reference'))
sys.path.insert(0, HERE)

import numpy as np
import torch

import stribor as st          # the reference
import cases
from make_golden import ref_layer


def _scatter(flat, ref_point, lower, upper, transformed):
    """flat searchsorted result over the in-box elements of `ref_point` -> [rows, dim] int32, -1 elsewhere"""
    pts = ref_point.reshape(-1, ref_point.shape[-1])
    inside = (pts >= lower) & (pts <= upper)
    assert int(inside.sum()) == flat.numel(), (int(inside.sum()), flat.numel())
    full = torch.full(pts.shape, -1, dtype=torch.int32)
    full[inside] = flat.to(torch.int32)
    full[:, ~transformed] = -1
    return full


def record_case(name):
    case = cases.build_bin_case(name)
    spec = case['spec']
    layers = [ref_layer(l) for l in spec]
    inp = case['inputs']
    kw = {k: inp[k] for k in ('latent', 't') if k in inp}
    x = inp['x']
    dim = x.shape[-1]
    out = {}
    capture = []
    orig = st.util.searchsorted

    def spy(knots, v, eps=1e-6):
        r = orig(knots, v, eps)
        capture.append(r.detach().clone())
        return r

    for i, (l, f) in enumerate(zip(spec, layers)):
        tr = l.get('transform')
        is_spline = tr is not None and tr['kind'] in ('quadratic', 'cubic')
        with torch.no_grad():
            if not is_spline:
                x = f(x, **kw)
                continue
            lower, upper = float(tr['lower']), float(tr['upper'])
            if l['type'] == 'coupling':
                m = st.util.get_mask(l['mask'])(dim)
                if m.numel() == 1 and dim != 1:
                    m = m.expand(dim)
                transformed = (m == 0)
            else:
                transformed = torch.ones(dim, dtype=torch.bool)
            st.util.searchsorted = spy
            try:
                capture.clear()
                y = f(x, **kw)
                fwd = _scatter(capture[0], x, lower, upper, transformed) if capture else \
                    torch.full((x.numel() // dim, dim), -1, dtype=torch.int32)
                capture.clear()
                xr, _ = f.inverse_and_log_det_jacobian(y, **kw)
                inv = _scatter(capture[0], y, lower, upper, transformed) if capture else torch.full_like(fwd, -1)
                # couplings re-evaluate the forward log-det at the recovered point (a second search); a bare
                # Spline uses the inverse map's own log-derivative (one search)
                fb = _scatter(capture[1], xr, lower, upper, transformed) if len(capture) > 1 else None
            finally:
                st.util.searchsorted = orig
            out[f'{name}|L{i}|x'] = x.numpy().copy()
            out[f'{name}|L{i}|y'] = y.numpy().copy()
            out[f'{name}|L{i}|xr'] = xr.numpy().copy()
            out[f'{name}|L{i}|fwd.bins'] = fwd.numpy()
            out[f'{name}|L{i}|inv.bins'] = inv.numpy()
            if fb is not None:
                out[f'{name}|L{i}|inv.fbins'] = fb.numpy()
            x = y
    return out


def stored_form(name, rec):
    """record_case(name) -> the arrays reference_bins.npz stores for the case (module docstring)"""
    layers = sorted({int(k.split('|')[1][1:]) for k in rec})
    rows = None
    if name in cases.BIN_CASES:
        n = rec[f'{name}|L{layers[0]}|x'].shape[0]
        rows = np.sort(np.random.RandomState(0).choice(n, n // 2, replace=False))
    pick = (lambda a: a) if rows is None else (lambda a: a[rows])
    out = {} if rows is None else {f'{name}|rows': rows}
    for i in layers:
        p = f'{name}|L{i}|'
        x = rec[p + 'x']
        if i > 0 and f'{name}|L{i - 1}|y' not in rec:
            out[p + 'x'] = pick(x)
        for k in ('y', 'xr'):
            out[p + k + '^x'] = pick(rec[p + k].view(np.int32) ^ x.view(np.int32))
        for k in ('fwd.bins', 'inv.bins', 'inv.fbins'):
            if p + k in rec:
                out[p + k] = pick(rec[p + k])
    return out


def main():
    blob = {}
    for name in cases.spline_cases():
        r = record_case(name)
        blob.update(stored_form(name, r))
        n_el = sum(int((v >= 0).sum()) for k, v in r.items() if k.endswith('fwd.bins'))
        print(name, len(r), 'arrays,', n_el, 'searched elements')
    path = os.path.join(HERE, 'reference_bins.npz')
    np.savez_compressed(path, **blob)
    print('wrote', path, len(blob), 'arrays', os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
