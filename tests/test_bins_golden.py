"""Bin-index parity, CPU part: the oracle's knot search reproduces the reference's recorded searchsorted
results bit for bit (tests/golden/reference_bins.npz, written by tests/golden/make_golden_bins.py from the
unmodified reference: util/search_sorted.py:3-5 via rational_quadratic_spline.py:194-197 and
cubic_spline.py:140-143)."""
import os

import numpy as np
import pytest
import torch

import cases
from oracle import coupling_flow_oracle as O

_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_bins.npz')
_BLOB = None


def bins_blob():
    global _BLOB
    if _BLOB is None:
        _BLOB = dict(np.load(_PATH))
    return _BLOB


def spline_layers(name):
    """[(layer index, layer spec)] of the spline layers of a case, with the case's extra inputs"""
    case = cases.build_bin_case(name)
    out = [(i, l) for i, l in enumerate(case['spec'])
           if l.get('transform', {}).get('kind') in ('quadratic', 'cubic')]
    return case, out


def recorded_layers(name):
    """-> (case, rows, [(layer index, layer spec, record)]) for the spline layers of a case, decoded from the
    compact stored form (make_golden_bins.stored_form).  A record holds numpy arrays: the layer input x, the
    reference's output y and its inverse xr of y, and its searches fwd.bins, inv.bins (and inv.fbins when
    recorded), over the recorded rows: `rows` indexes the case's rows, None when all of them are recorded."""
    case, layers = spline_layers(name)
    b = bins_blob()
    rows = b.get(f'{name}|rows')
    x = case['inputs']['x'].numpy()
    if rows is not None:
        x = x.reshape(-1, x.shape[-1])[rows]
    out = []
    for i, layer in layers:
        p = f'{name}|L{i}|'
        x = b.get(p + 'x', x)                   # else: the case input, or the previous spline layer's y
        bits = x.view(np.int32)
        rec = {'x': x, 'y': (bits ^ b[p + 'y^x']).view(np.float32), 'xr': (bits ^ b[p + 'xr^x']).view(np.float32)}
        rec.update({k: b[p + k] for k in ('fwd.bins', 'inv.bins', 'inv.fbins') if p + k in b})
        out.append((i, layer, rec))
        x = rec['y']
    return case, rows, out


@pytest.mark.parametrize('name', cases.spline_cases())
def test_oracle_bins_match_reference(name):
    case, _, layers = recorded_layers(name)
    latent = case['inputs'].get('latent')
    assert layers
    for i, layer, rec in layers:
        x = torch.from_numpy(rec['x'])
        y = torch.from_numpy(rec['y'])
        xr = torch.from_numpy(rec['xr'])
        lead = x.shape[:-1]
        want_f = torch.from_numpy(rec['fwd.bins']).long()
        got_f = O.layer_bins(layer, x, inverse=False, latent=latent).reshape(want_f.shape)
        assert torch.equal(got_f, want_f), f'{name} L{i}: forward bins differ'
        want_i = torch.from_numpy(rec['inv.bins']).long()
        got_i = O.layer_bins(layer, y, inverse=True, latent=latent).reshape(want_i.shape)
        assert torch.equal(got_i, want_i), f'{name} L{i}: inverse bins differ'
        if 'inv.fbins' in rec:
            want_r = torch.from_numpy(rec['inv.fbins']).long()
            got_r = O.layer_bins(layer, xr, inverse=False, latent=latent).reshape(want_r.shape)
            assert torch.equal(got_r, want_r), f'{name} L{i}: re-searched forward bins differ'
        # the recorded layer outputs are the oracle's too (same tolerance as test_oracle_golden)
        out, _ = O.layer_apply(layer, x, inverse=False, latent=latent)
        assert torch.allclose(out, y, rtol=1e-5, atol=1e-5)
        assert lead == y.shape[:-1]
