"""CPU: the oracle restatement vs the outputs recorded from the UNMODIFIED reference."""
import numpy as np
import pytest
import torch

import cases
from golden_util import blob, ref, has, pick
from oracle import coupling_flow_oracle as O

ALL = list(cases.CASES)


def _kw(inp, dtype):
    return {k: inp[k].to(dtype) for k in ('latent', 't') if k in inp}


@pytest.mark.parametrize('prec', ['f32', 'f64'])
@pytest.mark.parametrize('name', ALL)
def test_oracle_matches_reference(name, prec):
    dtype = torch.float32 if prec == 'f32' else torch.float64
    case = cases.build_case(name)
    spec = O.spec_to(case['spec'], dtype)
    inp = case['inputs']
    x = inp['x'].to(dtype)
    kw = _kw(inp, dtype)
    # same ATen kernels, same order of operations -> agreement to a few ulp
    tol = dict(rtol=2e-6, atol=2e-6) if prec == 'f32' else dict(rtol=1e-12, atol=1e-12)
    if 'cubic' in name and prec == 'f32':
        tol = dict(rtol=1e-4, atol=1e-4)    # one-root Cardano branch amplifies 1-ulp differences
    for op in case['ops']:
        if op == 'forward_ldj':
            y, ldj = O.flow_forward(spec, x, with_ldj=True, **kw)
            torch.testing.assert_close(y, ref(name, 'forward.y', prec), **tol)
            torch.testing.assert_close(ldj, ref(name, 'forward.ldj', prec), **tol)
        elif op == 'inverse_ldj':
            xr, ldj = O.flow_inverse(spec, x, with_ldj=True, **kw)
            torch.testing.assert_close(xr, ref(name, 'inverse.x', prec), **tol)
            torch.testing.assert_close(ldj, ref(name, 'inverse.ldj', prec), **tol)
        elif op == 'inverse_ldj_unit':
            y = ref(name, 'inverse_unit.y', prec)
            xr, ldj = O.flow_inverse(spec, y, with_ldj=True, **kw)
            torch.testing.assert_close(xr, ref(name, 'inverse_unit.x', prec), **tol)
            torch.testing.assert_close(ldj, ref(name, 'inverse_unit.ldj', prec), **tol)
        elif op == 'log_prob':
            lp = O.flow_log_prob(spec, x, **kw)
            torch.testing.assert_close(lp, ref(name, 'log_prob', prec), **tol)
        elif op == 'neural_flow':
            y = O.neural_flow_forward(spec, x, inp['t'].to(dtype))
            torch.testing.assert_close(y, ref(name, 'neural_flow.y', prec), **tol)
        elif op == 'neural_flow_t0':
            y = O.neural_flow_forward(spec, x, inp['t'].to(dtype), inp['t0'].to(dtype))
            torch.testing.assert_close(y, ref(name, 'neural_flow_t0.y', prec), **tol)
        elif op == 'nll_grad':
            params = []
            for l in spec:
                net = l['transform']['net'] if l['type'] != 'cont_affine_coupling' else l['net']
                for w, b in zip(net['weights'], net['biases']):
                    params += [w.requires_grad_(True), b.requires_grad_(True)]
            xg = x.clone().requires_grad_(True)
            loss = -O.flow_log_prob(spec, xg).mean()
            loss.backward()
            gt = dict(rtol=1e-3, atol=1e-5) if prec == 'f32' else dict(rtol=1e-9, atol=1e-11)
            torch.testing.assert_close(loss.detach(), ref(name, 'nll.loss', prec), **tol)
            torch.testing.assert_close(xg.grad, ref(name, 'nll.grad_x', prec), **gt)
            for i, p in enumerate(params):
                torch.testing.assert_close(pick(name, f'nll.grad_p{i}', p.grad), ref(name, f'nll.grad_p{i}', prec), **gt)


@pytest.mark.parametrize('name', [n for n in ALL if n.startswith('spline_')])
def test_oracle_bin_indices_exact(name):
    """Bin indices: bit-exact against the reference's own searchsorted calls."""
    case = cases.build_case(name)
    tr = case['spec'][0]['transform']
    x = case['inputs']['x']
    lat = case['inputs'].get('latent')
    p = O.transform_params(tr, lat, x.dtype)
    fn = O.rqs if tr['kind'] == 'quadratic' else O.cubic
    for inverse, key in ((False, 'forward.bins'), (True, 'inverse.bins')):
        if not has(name, key):
            continue
        _, _, bins = fn(x, p[0], p[1], p[2], inverse, tr['lower'], tr['upper'], return_bins=True)
        inside = (x >= tr['lower']) & (x <= tr['upper'])
        got = bins[inside]
        assert torch.equal(got, ref(name, key)), name


def test_reference_doc_example_golden_vector():
    """stribor/test/test_normalizing_flow.py:45-55 (== docstring flow.py:77-84)."""
    ls, sh = ref('doc_example', 'log_scale'), ref('doc_example', 'shift')
    spec = [{'type': 'elementwise',
             'transform': {'kind': 'affine', 'dim': 2, 'net': None, 'params': [ls, sh]}}]
    y = ref('doc_example', 'y')
    lp = O.flow_log_prob(spec, y)
    assert torch.allclose(lp, torch.tensor([[-1.7560], [-1.7434], [-2.1792]]), atol=1e-4)
    torch.testing.assert_close(lp, ref('doc_example', 'log_prob'), rtol=1e-6, atol=1e-6)
    z = ref('doc_example', 'z')
    torch.testing.assert_close(O.flow_forward(spec, z), ref('doc_example', 'forward_z'),
                               rtol=1e-6, atol=1e-6)


def test_masks_exact():
    """stribor/test/test_mask.py:4-30 plus the recorded vectors for larger dims."""
    assert O.make_mask('ordered_right_half', 5).tolist() == [0, 0, 1, 1, 1]
    assert O.make_mask('ordered_left_half', 5).tolist() == [1, 1, 0, 0, 0]
    assert O.make_mask('parity_even', 5).tolist() == [0, 1, 0, 1, 0]
    assert O.make_mask('parity_odd', 5).tolist() == [1, 0, 1, 0, 1]
    for k, v in blob().items():
        if k.startswith('mask|'):
            _, nm, d = k.split('|')
            assert np.array_equal(O.make_mask(nm, int(d)).numpy(), v), k
    with pytest.raises(NotImplementedError):
        O.make_mask('nope', 4)
