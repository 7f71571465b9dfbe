"""GPU: bin indices observed ON THE PRODUCT PATH (stb_layer_apply_bins) against the reference's recorded
searchsorted results (tests/golden/reference_bins.npz) -- BASELINE.json north_star: "bit-exact for ... spline
bin indices".  The instrumented call takes the same kernels as stb_layer_apply: the generic CUDA-core kernel,
the 256-row tcgen05 kernel (d <= 64, 16 bins, MLP[64]) and the 128-row one (d <= 128).

Policy: equality, except that an element whose input lies within a few ulp of a knot may land in the
ADJACENT bin (the knots themselves are fp32 results of a softmax + cumulative sum, SURVEY.md section 8c);
every such flip is checked to be adjacent and that close, and counted.  `python tests/test_gpu_bins.py`
prints the counts per case (the table in DESIGN.md section 5)."""
import os
import sys

import pytest
import torch

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (_ROOT, os.path.join(_ROOT, 'tests'), os.path.join(_ROOT, 'tests', 'golden')):     # `python tests/test_gpu_bins.py`
    if _p not in sys.path:
        sys.path.insert(0, _p)

import cases
from oracle import coupling_flow_oracle as O
from stribor_b200 import _lib, _ops
from stribor_b200.spec import layers_from_spec
from test_bins_golden import recorded_layers

pytestmark = pytest.mark.gpu
DEV = 'cuda'
FLIP_ULPS = 16          # a flipped element must be within this many ulp (of the box magnitude) of the knot


def _describe(module, dim, latent_dim):
    d = module.describe(dim, latent_dim, torch.device(DEV))
    return d


def cuda_bins(module, x, latent, direction):
    """(y, bins) of one layer through stb_layer_apply_bins, x [..., dim] on the GPU"""
    lead, dim = x.shape[:-1], x.shape[-1]
    d = _describe(module, dim, 0 if latent is None else latent.shape[-1])
    xf = x.reshape(-1, dim).contiguous()
    lf = None
    if latent is not None and d['meta'][2] > 0:
        lf = latent.expand(*lead, latent.shape[-1]).reshape(-1, latent.shape[-1]).contiguous()
    y, ldj, bins = _ops.layer_apply_bins(xf, lf, None, d['mask'], [p.detach() for p in d['params']], d.get('packed'),
                                         d['meta'], d['fmeta'], direction)
    L = _ops.make_struct(d['meta'], d['fmeta'], d['mask'], [p.detach() for p in d['params']], d.get('packed'))
    tensor_path = bool(_lib.lib().stb_layer_uses_tensor_path(L))
    return y.view(*lead, dim), bins, tensor_path


def compare_bins(got, want, layer, point, inverse, latent):
    """-> (n_searched, n_flips, max flip distance in ulp); asserts the flip policy"""
    want = want.to(got.device)
    assert got.shape == want.shape
    assert torch.equal(got < 0, want < 0), 'searched / not-searched pattern differs'
    diff = (got != want)
    n_flip = int(diff.sum())
    n = int((want >= 0).sum())
    worst = 0.0
    if n_flip:
        kn = O.layer_knots(layer, point.double().cpu(), inverse=inverse,
                           latent=None if latent is None else latent.double().cpu())
        kn = kn.reshape(-1, kn.shape[-2], kn.shape[-1])
        g, w = got.cpu().long(), want.cpu().long()
        idx = diff.cpu().nonzero()
        tr = layer['transform']
        mag = max(abs(float(tr['lower'])), abs(float(tr['upper'])))
        ulp = torch.finfo(torch.float32).eps * mag
        pts = point.reshape(-1, point.shape[-1]).double().cpu()
        for r, c in idx.tolist():
            assert abs(int(g[r, c]) - int(w[r, c])) == 1, f'non-adjacent bin flip at ({r},{c}): {g[r, c]} vs {w[r, c]}'
            knot = kn[r, c, max(int(g[r, c]), int(w[r, c]))]
            dist = abs(float(pts[r, c] - knot)) / ulp
            worst = max(worst, dist)
            assert dist <= FLIP_ULPS, f'bin flip {dist:.1f} ulp away from the knot at ({r},{c})'
    return n, n_flip, worst


def run_case(name):
    """-> list of per-layer dicts with the flip counts of the three searches"""
    case, rows, layers = recorded_layers(name)
    mods = [m.to(DEV) for m in layers_from_spec(case['spec'])]
    latent = case['inputs'].get('latent')
    lat_dev = None if latent is None else latent.to(DEV)
    # where only some rows of a case are recorded, the kernels still run on the whole batch (its tile shapes):
    # the recorded rows take their places in it, the others carry the kernels' own values, and the recorded
    # rows are compared
    whole = None if rows is None else case['inputs']['x'].to(DEV)
    rows = None if rows is None else torch.from_numpy(rows).to(DEV)

    def batch(v):
        v = torch.from_numpy(v).to(DEV)
        if rows is None:
            return v
        out = whole.clone()
        out[rows] = v
        return out

    def recorded(t):
        return t if rows is None else t[rows]

    out = []
    for i, layer, r in layers:
        mod = mods[i]
        x, y = torch.from_numpy(r['x']), torch.from_numpy(r['y'])
        rec = {'case': name, 'layer': i}
        # forward search at the layer input
        yc, fb, tp = cuda_bins(mod, batch(r['x']), lat_dev, _lib.FORWARD)
        whole = yc
        fb = recorded(fb)
        rec['tensor_path'] = tp
        rec['fwd'] = compare_bins(fb, torch.from_numpy(r['fwd.bins']), layer, x, False, latent)
        # inverse search at the reference's layer output
        xc, ib, _ = cuda_bins(mod, batch(r['y']), lat_dev, _lib.INVERSE)
        ib = recorded(ib)
        rec['inv'] = compare_bins(ib, torch.from_numpy(r['inv.bins']), layer, y, True, latent)
        # forward re-search at the RECOVERED point (what the reference does for the inverse log-det): the
        # kernels' own recovered x vs the reference's recorded re-search at its recovered x
        if 'inv.fbins' in r:
            _, rb, _ = cuda_bins(mod, xc, lat_dev, _lib.FORWARD)
            rb = recorded(rb)
            want = torch.from_numpy(r['inv.fbins']).to(DEV)
            same_pattern = torch.equal(rb < 0, want < 0)
            rec['refwd_flips'] = int((rb != want).sum()) if same_pattern else -1
            # the tensor-core kernels evaluate the inverse log-det in the bin the INVERSE search found instead of
            # re-searching (DESIGN 4.1): how often do the two differ?
            both = (ib >= 0) & (rb >= 0)
            rec['inv_vs_refwd'] = int(((ib != rb) & both).sum())
            rec['inv_vs_refwd_ref'] = int(((torch.from_numpy(r['inv.bins']).to(DEV) != want) & both).sum())
        out.append(rec)
    return out


@pytest.mark.parametrize('name', cases.spline_cases())
def test_cuda_bins_match_reference(name):
    for rec in run_case(name):
        # compare_bins has asserted the policy; fixtures small enough that any flip deserves a look are exact
        if not name.startswith('bins_'):
            assert rec['fwd'][1] == 0 and rec['inv'][1] == 0, rec


def test_tensor_path_is_observed():
    """the big fixtures really run on the tcgen05 kernels"""
    for name in ('bins_quadratic_d64_k16_h64', 'bins_cubic_d64_k16_h64', 'bins_quadratic_d128_k16_h64',
                 'bins_cubic_d128_k16_h64', 'bins_quadratic_d48_parity'):
        assert all(r['tensor_path'] for r in run_case(name)), name


@pytest.mark.parametrize('kind', ['quadratic', 'cubic'])
@pytest.mark.parametrize('dim', [64, 128])
def test_cuda_bins_match_oracle_large(kind, dim):
    """20 000 rows on the tensor-core kernels against the oracle's search on the oracle's own knots: equal
    except for adjacent flips within FLIP_ULPS of a knot (counted)."""
    rowsn = 20000
    case = cases._mk_flow(kind, dim, [64], 1, 16, rowsn, 900 + dim, lower=-4., upper=4., scale=1.6)()
    layer = case['spec'][0]
    mod = layers_from_spec(case['spec'])[0].to(DEV)
    x = case['inputs']['x']
    for inverse in (False, True):
        _, got, tp = cuda_bins(mod, x.to(DEV), None, _lib.INVERSE if inverse else _lib.FORWARD)
        assert tp
        want = O.layer_bins(layer, x, inverse=inverse).to(torch.int32)
        n, flips, worst = compare_bins(got, want, layer, x, inverse, None)
        assert n > 0.9 * rowsn * dim / 2
        assert flips <= 1e-4 * n, (flips, n)


if __name__ == '__main__':
    tot = {}
    print(f'{"case":38s} {"L":>2s} {"tc":>3s} {"searched":>9s} {"fwd flips":>9s} {"inv flips":>9s} {"max ulp":>8s} '
          f'{"refwd flips":>11s} {"inv!=refwd":>10s} {"(reference)":>11s}')
    for name in cases.spline_cases():
        for r in run_case(name):
            print(f'{name:38s} {r["layer"]:2d} {int(r["tensor_path"]):3d} {r["fwd"][0]:9d} {r["fwd"][1]:9d} {r["inv"][1]:9d} '
                  f'{max(r["fwd"][2], r["inv"][2]):8.1f} {r.get("refwd_flips", 0):11d} {r.get("inv_vs_refwd", 0):10d} '
                  f'{r.get("inv_vs_refwd_ref", 0):11d}')
            for k in ('fwd', 'inv'):
                tot[k] = tot.get(k, 0) + r[k][1]
            tot['n'] = tot.get('n', 0) + r['fwd'][0]
            tot['inv_vs_refwd'] = tot.get('inv_vs_refwd', 0) + r.get('inv_vs_refwd', 0)
    print('TOTAL', tot)
