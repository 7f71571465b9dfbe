"""GPU: flows in float64 -- the double CUDA-core kernels against the oracle evaluated in float64
(``O.spec_to(spec, torch.float64)``): values, bin indices, gradients (``torch.autograd.gradcheck`` and fp64
autograd through the oracle) and a float64 training session."""
import contextlib

import pytest
import torch
from torch.func import functional_call

import cases
from golden_util import ref
from oracle import coupling_flow_oracle as O
import stribor_b200 as st
from stribor_b200 import _lib, _ops
from stribor_b200.spec import layers_from_spec

pytestmark = pytest.mark.gpu
DEV = 'cuda'


def _tol(name):
    return 1e-9 if 'cubic' in name else 1e-10


def _close(got, want, tol, what):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err = (got - want).abs()
    bad = err > tol + tol * want.abs()
    assert not bool(bad.any()), \
        f'{what}: {int(bad.sum())} of {bad.numel()} outside rtol = atol = {tol:g}, max abs err {float(err.max()):.3e}'


def _flow64(case):
    layers = [l.to(DEV).double() for l in layers_from_spec(case['spec'])]
    return st.NormalizingFlow(st.UnitNormal(case['inputs']['x'].shape[-1]), layers), layers


@pytest.mark.parametrize('name', list(cases.CASES))
@pytest.mark.parametrize('fused', [True, False])
def test_values_match_fp64_oracle(name, fused):
    case = cases.build_case(name)
    if all(op == 'nll_grad' for op in case['ops']):
        pytest.skip('gradient case')
    spec = O.spec_to(case['spec'], torch.float64)
    flow, layers = _flow64(case)
    inp = case['inputs']
    x = inp['x'].double()
    kw = {k: inp[k].double() for k in ('latent', 't') if k in inp}
    kwd = {k: v.to(DEV) for k, v in kw.items()}
    tol = _tol(name)
    if not fused:
        for p in flow.parameters():
            p.requires_grad_(True)                  # the layer-by-layer, autograd-capable path
    with torch.no_grad() if fused else contextlib.nullcontext():
        for op in case['ops']:
            if op == 'forward_ldj':
                y, ldj = flow.forward_and_log_det_jacobian(x.to(DEV), **kwd)
                wy, wl = O.flow_forward(spec, x, with_ldj=True, **kw)
                _close(y, wy, tol, 'forward.y')
                _close(ldj, wl, tol, 'forward.ldj')
                assert torch.equal(flow.forward(x.to(DEV), **kwd), y)
            elif op in ('inverse_ldj', 'inverse_ldj_unit'):
                yin = x if op == 'inverse_ldj' else ref(name, 'inverse_unit.y').double()
                xr, ldj = flow.inverse_and_log_det_jacobian(yin.to(DEV), **kwd)
                wx, wl = O.flow_inverse(spec, yin, with_ldj=True, **kw)
                _close(xr, wx, tol, f'{op}.x')
                _close(ldj, wl, tol, f'{op}.ldj')
            elif op == 'log_prob':
                _close(flow.log_prob(x.to(DEV), **kwd), O.flow_log_prob(spec, x, **kw), tol, 'log_prob')
            elif op in ('neural_flow', 'neural_flow_t0'):
                t0 = inp['t0'].double() if op == 'neural_flow_t0' else None
                got = st.NeuralFlow(layers)(x.to(DEV), t=inp['t'].double().to(DEV),
                                            t0=None if t0 is None else t0.to(DEV))
                _close(got, O.neural_flow_forward(spec, x, inp['t'].double(), t0), tol, op)
    assert all(p.dtype == torch.float64 for p in flow.parameters())


@pytest.mark.parametrize('name', ['spline_quadratic_7x4x5_k10_l13', 'spline_cubic_7x4x5_k10_l0',
                                  'quadratic_d5_parity', 'cubic_d7_ordered', 'quadratic_d16_default_box',
                                  'cubic_d16_default_box'])
@pytest.mark.parametrize('inverse', [False, True])
def test_bins_match_searchsorted_on_fp64_knots(name, inverse):
    """stb_layer_apply_bins in float64 == searchsorted on the oracle's float64 knots, except within 1e-12 of a knot"""
    case = cases.build_case(name)
    layer = O.spec_to(case['spec'], torch.float64)[0]
    module = layers_from_spec(case['spec'])[0].to(DEV).double()
    x = case['inputs']['x'].double()
    lat = case['inputs'].get('latent')
    lat = None if lat is None else lat.double().expand(*x.shape[:-1], lat.shape[-1])
    dim = x.shape[-1]
    d = module.describe(dim, 0 if lat is None else lat.shape[-1], torch.device(DEV))
    xf = x.reshape(-1, dim).contiguous()
    lf = None if (lat is None or d['meta'][2] == 0) else lat.reshape(-1, lat.shape[-1]).contiguous().to(DEV)
    _, _, bins = _ops.layer_apply_bins(xf.to(DEV), lf, None, d['mask'], [p.detach() for p in d['params']], None,
                                       d['meta'], d['fmeta'], _lib.INVERSE if inverse else _lib.FORWARD)
    want = O.layer_bins(layer, x, inverse=inverse, latent=lat).reshape(-1, dim)
    got = bins.cpu().long()
    assert torch.equal(got < 0, want < 0)
    diff = (got != want).nonzero().tolist()
    if diff:
        kn = O.layer_knots(layer, x, inverse=inverse, latent=lat).reshape(-1, dim, layer['transform']['n_bins'] + 1)
        for r, c in diff:
            knot = kn[r, c, max(int(got[r, c]), int(want[r, c]))]
            assert abs(float(xf[r, c] - knot)) <= 1e-12, (r, c, int(got[r, c]), int(want[r, c]))


class _Method(torch.nn.Module):
    """``module.<method>`` as a forward, so that torch.func.functional_call can swap the parameters in"""

    def __init__(self, module, method):
        super().__init__()
        self.m, self.method = module, method

    def forward(self, *args, **kwargs):
        return getattr(self.m, self.method)(*args, **kwargs)


def _gradcheck(module, method, inputs, **kwargs):
    """gradcheck of ``module.method(*inputs, **kwargs)`` wrt the inputs AND every parameter of the module"""
    wrap = _Method(module, method)
    names = [n for n, _ in wrap.named_parameters()]
    params = [p.detach().clone().requires_grad_(True) for _, p in wrap.named_parameters()]
    n_in = len(inputs)

    def fn(*args):
        return functional_call(wrap, dict(zip(names, args[n_in:])), args[:n_in], kwargs)

    assert torch.autograd.gradcheck(fn, tuple(v.requires_grad_(True) for v in inputs) + tuple(params))


def _coupling(kind, dim, n_bins=5):
    if kind == 'affine':
        tr = st.Affine(dim, latent_net=st.net.MLP(dim, [8], 2 * dim))
    else:
        P = 2 * n_bins + (n_bins - 1 if kind == 'quadratic' else 2)
        tr = st.Spline(dim, n_bins, latent_net=st.net.MLP(dim, [8], dim * P), lower=-3., upper=3., spline_type=kind)
    return st.Coupling(tr, 'ordered_right_half')


@pytest.mark.parametrize('kind', ['quadratic', 'cubic', 'affine'])
@pytest.mark.parametrize('method', ['forward_and_log_det_jacobian', 'inverse_and_log_det_jacobian'])
def test_gradcheck_coupling(kind, method):
    torch.manual_seed(3)
    m = _coupling(kind, 4).to(DEV).double()
    x = torch.rand(5, 4, dtype=torch.float64, device=DEV) * 4 - 2
    _gradcheck(m, method, (x,))


@pytest.mark.parametrize('method', ['forward_and_log_det_jacobian', 'inverse_and_log_det_jacobian'])
def test_gradcheck_continuous_affine(method):
    torch.manual_seed(4)
    m = st.ContinuousAffineCoupling(st.net.MLP(4 + 1, [8], 8), st.net.TimeLinear(8), 'ordered_left_half')
    m = m.to(DEV).double()
    x = torch.randn(5, 4, dtype=torch.float64, device=DEV)
    t = torch.rand(5, 1, dtype=torch.float64, device=DEV)
    _gradcheck(m, method, (x,), t=t)


def _spline_inputs(kind, K, n_der, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(6, 3, generator=g, dtype=torch.float64) * 5 - 2.5           # [-2.5, 2.5] in the box [-3, 3]
    w, h = (torch.randn(6, 3, K, generator=g, dtype=torch.float64) for _ in range(2))
    d = torch.randn(6, 3, n_der, generator=g, dtype=torch.float64)
    return [v.to(DEV) for v in (x, w, h, d)]


@pytest.mark.parametrize('kind, opts, extra', [
    ('quadratic', {}, -1), ('quadratic', {'min_bin_width': 1e-2, 'min_bin_height': 2e-2, 'min_derivative': 1e-4}, -1),
    ('quadratic', {}, 1), ('quadratic', {'min_bin_width': 1e-2, 'min_derivative': 1e-2}, 1),
    ('cubic', {}, 0), ('cubic', {'min_bin_width': 2e-2, 'min_bin_height': 3e-2, 'eps': 1e-4,
                                 'quadratic_threshold': 1e-2}, 0)])
@pytest.mark.parametrize('inverse', [False, True])
def test_gradcheck_functional_splines(kind, opts, extra, inverse):
    """both functional splines, with and without options, with K - 1 and K + 1 derivatives"""
    K = 5
    x, w, h, d = _spline_inputs(kind, K, K + extra if kind == 'quadratic' else 2, 7)
    fn = st.util.unconstrained_rational_quadratic_spline if kind == 'quadratic' else st.util.unconstrained_cubic_spline
    f = lambda *a: fn(*a, inverse=inverse, lower=-3., upper=3., **opts)
    assert torch.autograd.gradcheck(f, tuple(v.requires_grad_(True) for v in (x, w, h, d)))
    if not opts and extra != 1:
        # defaults: the fp64 oracle's values as well.  (K + 1 derivatives travel as spline options, whose minimums
        # are float in both dtypes: 1e-3 arrives as float(1e-3) = 1.0000000475e-3, a 5e-11 relative change.)
        o = (O.rqs if kind == 'quadratic' else O.cubic)(x.cpu(), w.cpu(), h.cpu(), d.cpu(), inverse, -3., 3.)
        y, ld = f(x, w, h, d)
        _close(y, o[0], _tol(kind), 'functional out')
        _close(ld, o[1], _tol(kind), 'functional log-diag')


@pytest.mark.parametrize('kind', ['quadratic', 'cubic', 'affine'])
def test_gradcheck_flow_log_prob(kind):
    torch.manual_seed(5)
    flow = st.NormalizingFlow(st.UnitNormal(4), [_coupling(kind, 4, n_bins=3) for _ in range(2)] +
                              [st.Flip(), _coupling(kind, 4, n_bins=3)]).to(DEV).double()
    x = torch.rand(4, 4, dtype=torch.float64, device=DEV) * 4 - 2
    _gradcheck(flow, 'log_prob', (x,))


@pytest.mark.parametrize('name', [n for n in cases.CASES if n.startswith('grad_')])
def test_nll_gradients_match_fp64_oracle_autograd(name):
    case = cases.build_case(name)
    spec = O.spec_to(case['spec'], torch.float64)
    leaves = []
    for layer in spec:
        for w, b in zip(layer['transform']['net']['weights'], layer['transform']['net']['biases']):
            leaves += [w.requires_grad_(True), b.requires_grad_(True)]
    x64 = case['inputs']['x'].double().requires_grad_(True)
    (-O.flow_log_prob(spec, x64).mean()).backward()
    flow, _ = _flow64(case)
    x = case['inputs']['x'].double().to(DEV).requires_grad_(True)
    loss = -flow.log_prob(x).mean()
    loss.backward()
    _close(x.grad, x64.grad, 1e-9, 'grad_x')
    got = list(flow.parameters())
    assert len(got) == len(leaves)
    for i, (p, r) in enumerate(zip(got, leaves)):
        _close(p.grad, r.grad, 1e-9, f'grad of parameter {i}')


def _headline(kind, dim=64):
    P = 47 if kind == 'quadratic' else 34
    masks = ('ordered_right_half', 'ordered_left_half')
    return st.NormalizingFlow(st.UnitNormal(dim), [
        st.Coupling(st.Spline(dim, 16, latent_net=st.net.MLP(dim, [64], dim * P), lower=-4., upper=4.,
                              spline_type=kind), masks[i % 2]) for i in range(8)])


@pytest.mark.parametrize('kind', ['quadratic', 'cubic'])
def test_float64_training_session(kind):
    """set_default_dtype(float64): build, sample, log_prob, one optimizer step, then the round trip"""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        torch.manual_seed(6)
        flow = _headline(kind).to(DEV)
        assert all(p.dtype == torch.float64 for p in flow.parameters())
        opt = torch.optim.Adam(flow.parameters(), lr=1e-3)
        x = flow.sample(512).detach()
        assert x.dtype == torch.float64 and x.shape == (512, 64)
        loss = -flow.log_prob(x).mean()
        loss.backward()
        assert all(p.grad is not None and bool(torch.isfinite(p.grad).all()) for p in flow.parameters())
        opt.step()
        with torch.no_grad():
            lp = flow.log_prob(x)
            _close(lp, O.flow_log_prob(st.spec.spec_from_layers(list(flow.transforms)), x.cpu()), _tol(kind),
                   'log_prob after the step')
            xr = flow.inverse(flow.forward(x))
            tol = 1e-8 if kind == 'cubic' else 1e-10
            # An element may exceed the bound only where the float64 oracle's own round trip on the same
            # parameters is that far off too: the cubic inverse's one-root (Cardano) branch cancels p + q
            # when the discriminant is near 0 and amplifies rounding there, in any implementation.
            spec = st.spec.spec_from_layers(list(flow.transforms))
            own = (O.flow_inverse(spec, O.flow_forward(spec, x.cpu())) - x.cpu()).abs()
            err = (xr.cpu() - x.cpu()).abs()
            bad = (err > tol + tol * x.cpu().abs()) & (err > 4 * own + tol)
            assert not bool(bad.any()), f'inverse(forward(x)): {int(bad.sum())} elements, max abs err {float(err.max()):.3e}'
    finally:
        torch.set_default_dtype(old)


def test_double_switches_a_cached_flow_and_mixed_dtypes_raise():
    case = cases.build_case('quadratic_d5_parity')
    layers = [l.to(DEV) for l in layers_from_spec(case['spec'])]
    flow = st.NormalizingFlow(st.UnitNormal(5), layers)
    x = case['inputs']['x'].to(DEV)
    with torch.no_grad():
        flow.log_prob(x)                                   # a float32 call plan is cached
        with pytest.raises(TypeError):
            flow.log_prob(x.double())                      # float32 weights, float64 input: not promoted
        flow.double()
        lp = flow.log_prob(x.double())
        assert lp.dtype == torch.float64
        _close(lp, O.flow_log_prob(O.spec_to(case['spec'], torch.float64), x.cpu().double()), 1e-10, 'log_prob')
        with pytest.raises(TypeError):
            flow.log_prob(x)
        with pytest.raises(TypeError):
            st.util.unconstrained_cubic_spline(x.double(), *(torch.zeros(*x.shape, k, device=DEV) for k in (3, 3, 2)))


def test_set_data_coupling():
    """set_data: the selected rows of each set go through a 'none'-mask coupling of the same transform"""
    torch.manual_seed(8)
    tr = st.Spline(3, 4, latent_net=st.net.MLP(3, [8], 3 * 11), lower=-3., upper=3., spline_type='quadratic')
    c = st.Coupling(tr, 'ordered_right_half', set_data=True).to(DEV).double()
    x = torch.randn(2, 6, 3, dtype=torch.float64, device=DEV)
    with torch.no_grad():
        y, ldj = c.forward_and_log_det_jacobian(x)
        sel = (c.mask_func(6) == 0).nonzero().view(-1).to(DEV)
        ref_layer = O.spec_to(st.spec.spec_from_layers([st.Coupling(tr, 'none')]), torch.float64)[0]
        want, wl = O.layer_apply(ref_layer, x.index_select(-2, sel).cpu(), inverse=False)
        _close(y.index_select(-2, sel), want, 1e-10, 'set_data y')
        _close(ldj.index_select(-2, sel), wl, 1e-10, 'set_data ldj')
        keep = [i for i in range(6) if i not in sel.tolist()]
        assert torch.equal(y[:, keep], x[:, keep])
