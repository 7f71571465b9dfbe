"""The functional spline API's options: minimum bin width / height, minimum derivative and free boundary
derivatives (K + 1 derivative parameters) of unconstrained_rational_quadratic_spline, and the minimum bin sizes,
root window `eps` and `quadratic_threshold` of unconstrained_cubic_spline.  Values and gradients against the
fp32 / fp64 oracle, bit-exact identities between equivalent calls, the reference's own property checkers on a
Spline subclass that passes an option, and the errors.  The host-side tests at the end need no GPU."""
import contextlib
import ctypes as C
import importlib.util
import math
import os
import sys

import numpy as np
import pytest
import torch

from golden_util import close_or_arbitrated
from oracle import coupling_flow_oracle as O
import stribor_b200 as st
from stribor_b200 import _lib, _ops
from stribor_b200.util import splines as SP
from test_gpu_grad import _assert_grad_close

DEV = 'cuda'
gpu = pytest.mark.gpu
RQS = st.util.unconstrained_rational_quadratic_spline
CUB = st.util.unconstrained_cubic_spline
ROWS, DIM = 1000, 4
LO, HI = -2.0, 2.0
BOX = dict(left=-1., right=1., bottom=-3., top=2.)


@contextlib.contextmanager
def _oracle_constants(**consts):
    """The oracle's rqs / cubic read their spline constants (RQS_MIN_W, CUB_EPS, ...) from module globals when
    called: evaluate it with other values by setting them for the duration of the call."""
    old = {k: getattr(O, k) for k in consts}
    for k, v in consts.items():
        setattr(O, k, v)
    try:
        yield
    finally:
        for k, v in old.items():
            setattr(O, k, v)


def oracle_rqs(x, uw, uh, ud, inverse, lower, upper, min_bin_width=1e-3, min_bin_height=1e-3,
               min_derivative=1e-3, **box):
    """O.rqs with the reference's keyword options; `ud` may hold K - 1 or K + 1 derivatives."""
    with _oracle_constants(RQS_MIN_W=min_bin_width, RQS_MIN_H=min_bin_height, RQS_MIN_D=min_derivative):
        return O.rqs(x, uw, uh, ud, inverse, lower, upper, **box)


def oracle_cubic(x, uw, uh, ud, inverse, lower, upper, min_bin_width=1e-2, min_bin_height=1e-2, eps=1e-5,
                 quadratic_threshold=1e-3):
    """O.cubic with the reference's keyword options."""
    with _oracle_constants(CUB_MIN_W=min_bin_width, CUB_MIN_H=min_bin_height, CUB_EPS=eps,
                           CUB_QUAD_THRESHOLD=quadratic_threshold):
        return O.cubic(x, uw, uh, ud, inverse, lower, upper)


def _edge(md):
    """Pad value of the K - 1 derivative layout: log(exp(1 - min_derivative) - 1) of the float32 minimum,
    evaluated in double and rounded once."""
    return float(np.float32(math.log(math.exp(1.0 - float(np.float32(md))) - 1.0)))


def _inputs(lo, hi, seed, rows=ROWS, dim=DIM):
    """Uniform over the box and half a unit beyond it on both sides, with whole rows exactly on the box
    edges and deep in the tails."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(rows, dim, generator=g) * (hi - lo + 1.0) + (lo - 0.5)
    x[0], x[1], x[2], x[3] = lo, hi, lo - 3.0, hi + 3.0
    return x


def _params(K, n_der, seed, rows=ROWS, dim=DIM):
    """Unit-scale parameters: no bin so flat that fp32 rounding of y alone moves the inverse by 1e-4."""
    g = torch.Generator().manual_seed(seed)
    uw = torch.randn(rows, dim, K, generator=g)
    uh = torch.randn(rows, dim, K, generator=g)
    ud = torch.randn(rows, dim, n_der, generator=g)
    return uw, uh, ud


def _dev(*ts):
    return [t.to(DEV) for t in ts]


def _check(got, o32, o64, what, frac=0.0, atol=1e-5):
    """The fp64-arbitrated rule at rtol = 1e-5 and `atol`; where the fp64 oracle is not finite (the cubic inverse
    of a bin with a = b = 0 is 0/0 in the reference too) nothing is compared."""
    fin = torch.isfinite(o64)
    fail, _, mx = close_or_arbitrated(got.cpu()[fin], o32[fin], o64[fin], 1e-5, atol)
    assert fail <= frac, f'{what}: {fail:.3%} outside tolerance, max abs err {mx:.3e}'


# Tolerances of the value tests.  The kernels form the knots with a float running sum, where the oracle's CPU
# cumsum accumulates in double, so a knot can sit a few ulp away from the oracle's; that moves an output by up to
# ~2.5e-5 in rare elements and, through theta = (x - x_k) / w_k in a narrow bin, the log-derivative by up to ~1e-3
# at K = 16 / 33.  The reference defaults, which run the kernels unchanged, show the same errors: rtol = atol =
# 1e-5 with one outlier in a thousand for outputs, atol = 2e-3 for log-derivatives.
OUT_FRAC = 1e-3
LD_ATOL = 2e-3


def _box_kw(box):
    return dict(BOX) if box else {}


def _dir_range(box, inverse):
    if not box:
        return LO, HI
    return (BOX['bottom'], BOX['top']) if inverse else (BOX['left'], BOX['right'])


RQS_OPTS = {
    'defaults': ({}, False),
    'min_sizes_1_over_K': ('1/K', False),
    'tiny_minima': (dict(min_bin_width=1e-6, min_bin_height=1e-6, min_derivative=1e-6), False),
    'min_derivative_1e-5': (dict(min_derivative=1e-5), False),
    'min_derivative_0.1': (dict(min_derivative=0.1), False),
    'free_edges': ({}, True),
    'free_edges_custom': (dict(min_bin_width=2e-2, min_bin_height=1e-4, min_derivative=0.1), True),
}


def _rqs_opts(name, K):
    opts, free = RQS_OPTS[name]
    if opts == '1/K':
        opts = dict(min_bin_width=1.0 / K, min_bin_height=1.0 / K)
    return dict(opts), free


# ------------------------------------------------------------------------------------------------------------
# values
# ------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize('K', [1, 3, 16, 33])
@pytest.mark.parametrize('opt', list(RQS_OPTS))
@pytest.mark.parametrize('box', [False, True])
def test_rqs_options_match_oracle(K, opt, box):
    opts, free = _rqs_opts(opt, K)
    uw, uh, ud = _params(K, K + 1 if free else K - 1, seed=K)
    p64 = [p.double() for p in (uw, uh, ud)]
    with torch.no_grad():
        for inverse in (False, True):
            lo, hi = _dir_range(box, inverse)
            x = _inputs(lo, hi, seed=10 * K + inverse)
            y, ld = RQS(*_dev(x, uw, uh, ud), inverse=inverse, lower=LO, upper=HI, **_box_kw(box), **opts)
            o32, l32 = oracle_rqs(x, uw, uh, ud, inverse, LO, HI, **_box_kw(box), **opts)
            o64, l64 = oracle_rqs(x.double(), *p64, inverse, LO, HI, **_box_kw(box), **opts)
            what = f'rqs K={K} {opt} box={box} inverse={inverse}'
            _check(y, o32, o64, what + ' out', OUT_FRAC)
            _check(ld, l32, l64, what + ' log-derivative', atol=LD_ATOL)
            tail = (x < lo) | (x > hi)
            assert torch.equal(y.cpu()[tail], x[tail]) and bool((ld.cpu()[tail] == 0).all())


CUB_OPTS = {
    'defaults': {},
    'min_sizes_1_over_K': '1/K',
    'tiny_minima': dict(min_bin_width=1e-6, min_bin_height=1e-6),
    'wide_eps_threshold': dict(eps=1e-3, quadratic_threshold=1e-2),
    'narrow_eps_threshold': dict(min_bin_width=2e-2, min_bin_height=1e-4, eps=1e-7, quadratic_threshold=1e-5),
}


def _cub_opts(name, K):
    opts = CUB_OPTS[name]
    return dict(min_bin_width=1.0 / K, min_bin_height=1.0 / K) if opts == '1/K' else dict(opts)


@gpu
@pytest.mark.parametrize('K', [1, 3, 16, 33])
@pytest.mark.parametrize('opt', list(CUB_OPTS))
def test_cubic_options_match_oracle(K, opt):
    opts = _cub_opts(opt, K)
    uw, uh, ud = _params(K, 2, seed=K)
    p64 = [p.double() for p in (uw, uh, ud)]
    with torch.no_grad():
        for inverse in (False, True):
            x = _inputs(LO, HI, seed=10 * K + inverse)
            y, ld = CUB(*_dev(x, uw, uh, ud), inverse=inverse, lower=LO, upper=HI, **opts)
            o32, l32 = oracle_cubic(x, uw, uh, ud, inverse, LO, HI, **opts)
            o64, l64 = oracle_cubic(x.double(), *p64, inverse, LO, HI, **opts)
            # the inverse's root selection amplifies 1-ulp differences in the bin coefficients: the same outlier
            # bound as the other cubic inverse tests
            frac = 2e-3 if inverse else 0.0
            what = f'cubic K={K} {opt} inverse={inverse}'
            _check(y, o32, o64, what + ' out', max(frac, OUT_FRAC))
            _check(ld, l32, l64, what + ' log-derivative', frac, LD_ATOL)
            tail = (x < LO) | (x > HI)
            assert torch.equal(y.cpu()[tail], x[tail]) and bool((ld.cpu()[tail] == 0).all())


# ------------------------------------------------------------------------------------------------------------
# gradients
# ------------------------------------------------------------------------------------------------------------
def _loss(out, ld):
    return out.sin().sum() + (ld * ld).sum() + ld.sum()


def _grads(fn, x, params, inverse, **kw):
    leaves = [t.clone().requires_grad_(True) for t in (x, *params)]
    out, ld = fn(leaves[0], *leaves[1:], inverse=inverse, lower=LO, upper=HI, **kw)
    _loss(out, ld).backward()
    return [t.grad for t in leaves]


@gpu
@pytest.mark.parametrize('K', [3, 16])
@pytest.mark.parametrize('opt', ['min_sizes_1_over_K', 'tiny_minima', 'min_derivative_1e-5', 'free_edges',
                                 'free_edges_custom'])
@pytest.mark.parametrize('inverse', [False, True])
def test_rqs_option_gradients_match_oracle_autograd(K, opt, inverse):
    opts, free = _rqs_opts(opt, K)
    uw, uh, ud = _params(K, K + 1 if free else K - 1, seed=100 + K)
    x = _inputs(LO, HI, seed=200 + K)
    got = _grads(RQS, *_dev(x), _dev(uw, uh, ud), inverse, **opts)
    r32 = _grads(oracle_rqs, x, (uw, uh, ud), inverse, **opts)
    r64 = _grads(oracle_rqs, x.double(), [p.double() for p in (uw, uh, ud)], inverse, **opts)
    for name, g, a, b in zip(('inputs', 'widths', 'heights', 'derivatives'), got, r32, r64):
        _assert_grad_close(g, a, b, f'rqs K={K} {opt} inverse={inverse}: gradient wrt {name}')
    tail = (x < LO) | (x > HI)
    for g in got[1:]:
        assert bool((g.cpu()[tail] == 0).all()), 'tail elements must give zero parameter gradients'
    if free:                                   # the boundary derivative parameters are learned too
        assert bool((got[3][..., 0] != 0).any()) and bool((got[3][..., -1] != 0).any())


@gpu
@pytest.mark.parametrize('K', [3, 16])
@pytest.mark.parametrize('opt', ['tiny_minima', 'wide_eps_threshold', 'narrow_eps_threshold'])
@pytest.mark.parametrize('inverse', [False, True])
def test_cubic_option_gradients_match_oracle_autograd(K, opt, inverse):
    opts = _cub_opts(opt, K)
    uw, uh, ud = _params(K, 2, seed=100 + K)
    x = _inputs(LO, HI, seed=200 + K)
    got = _grads(CUB, *_dev(x), _dev(uw, uh, ud), inverse, **opts)
    r32 = _grads(oracle_cubic, x, (uw, uh, ud), inverse, **opts)
    r64 = _grads(oracle_cubic, x.double(), [p.double() for p in (uw, uh, ud)], inverse, **opts)
    for name, g, a, b in zip(('inputs', 'widths', 'heights', 'derivatives'), got, r32, r64):
        _assert_grad_close(g, a, b, f'cubic K={K} {opt} inverse={inverse}: gradient wrt {name}')
    tail = (x < LO) | (x > HI)
    for g in got[1:]:
        assert bool((g.cpu()[tail] == 0).all()), 'tail elements must give zero parameter gradients'


# ------------------------------------------------------------------------------------------------------------
# bit-exact identities
# ------------------------------------------------------------------------------------------------------------
def _run_with_grads(fn, x, params, inverse, **kw):
    leaves = [t.clone().requires_grad_(True) for t in (x, *params)]
    out, ld = fn(leaves[0], *leaves[1:], inverse=inverse, lower=LO, upper=HI, **kw)
    _loss(out, ld).backward()
    return [out.detach(), ld.detach()] + [t.grad for t in leaves]


@gpu
@pytest.mark.parametrize('inverse', [False, True])
def test_explicit_defaults_equal_omitted(inverse):
    x = _inputs(LO, HI, seed=7).to(DEV)
    for fn, n_der, defaults in ((RQS, 15, dict(min_bin_width=1e-3, min_bin_height=1e-3, min_derivative=1e-3)),
                                (CUB, 2, dict(min_bin_width=1e-2, min_bin_height=1e-2, eps=1e-5,
                                              quadratic_threshold=1e-3))):
        params = _dev(*_params(16, n_der, seed=8))
        a = _run_with_grads(fn, x, params, inverse)
        b = _run_with_grads(fn, x, params, inverse, **defaults)
        for u, v in zip(a, b):
            assert torch.equal(u, v)


def _forced_runtime(kind, x, params, inverse, opts):
    """The kernels instantiated for run-time options, fed the default values."""
    fmeta = [LO, HI] * 3 + [1.] + list(opts)
    return SP._row_params_call(kind, x, params, params[0].shape[-1], inverse, fmeta, False)


@gpu
@pytest.mark.parametrize('inverse', [False, True])
def test_runtime_option_kernels_reproduce_the_compiled_defaults(inverse):
    x = _inputs(LO, HI, seed=9).to(DEV)
    for fn, kind, n_der, opts in ((RQS, _lib.RQS, 15, (1e-3, 1e-3, 1e-3, 0., 0., 0.)),
                                  (CUB, _lib.CUBIC, 2, (1e-2, 1e-2, 0., 0., 1e-5, 1e-3))):
        params = _dev(*_params(16, n_der, seed=10))
        want = _run_with_grads(fn, x, params, inverse)
        got = _run_with_grads(lambda *a, inverse, lower, upper: _forced_runtime(kind, a[0], list(a[1:]), inverse, opts),
                              x, params, inverse)
        for u, v in zip(want, got):
            assert torch.equal(u, v)


@gpu
@pytest.mark.parametrize('md', [1e-3, 1e-5, 0.1])
@pytest.mark.parametrize('K', [1, 16])
@pytest.mark.parametrize('inverse', [False, True])
def test_k_minus_1_derivatives_equal_padded_k_plus_1(md, K, inverse):
    uw, uh, ud = _params(K, K - 1, seed=11)
    pad = torch.full(ud.shape[:-1] + (1,), _edge(md))
    ud_full = torch.cat([pad, ud, pad], -1)
    x = _inputs(LO, HI, seed=12).to(DEV)
    a = _run_with_grads(RQS, x, _dev(uw, uh, ud), inverse, min_derivative=md)
    b = _run_with_grads(RQS, x, _dev(uw, uh, ud_full), inverse, min_derivative=md)
    for u, v in zip(a[:5], b[:5]):                      # outputs, log-derivatives, inputs / widths / heights grads
        assert torch.equal(u, v)
    assert torch.equal(a[5], b[5][..., 1:-1])           # interior derivative gradients


# ------------------------------------------------------------------------------------------------------------
# properties
# ------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize('opt', ['min_sizes_1_over_K', 'tiny_minima', 'min_derivative_1e-5', 'min_derivative_0.1',
                                 'free_edges_custom'])
def test_rqs_round_trip_and_log_derivative_vs_autograd(opt):
    K = 16
    opts, free = _rqs_opts(opt, K)
    uw, uh, ud = _dev(*_params(K, K + 1 if free else K - 1, seed=13))
    x = _inputs(LO, HI, seed=14).to(DEV).requires_grad_(True)
    y, ld = RQS(x, uw, uh, ud, lower=LO, upper=HI, **opts)
    xr, ldr = RQS(y.detach(), uw, uh, ud, inverse=True, lower=LO, upper=HI, **opts)
    # the reference checkers' allclose(atol=1e-4); a bin with slope ~1e-3 turns the rounding of y alone into an
    # error above that in x, and bins a few 1e-6 wide (minima 1e-6) shift the log-derivative of the recovered point,
    # so a few elements in a thousand may exceed it
    assert (~torch.isclose(xr, x.detach(), rtol=1e-5, atol=1e-4)).float().mean().item() <= 1e-3
    assert (~torch.isclose(ldr, -ld.detach(), rtol=1e-5, atol=1e-4)).float().mean().item() <= 5e-3
    dydx, = torch.autograd.grad(y.sum(), x)         # element-wise: the Jacobian is diagonal
    torch.testing.assert_close(dydx.log(), ld.detach(), rtol=0, atol=1e-4)


@gpu
@pytest.mark.parametrize('opt', ['tiny_minima', 'wide_eps_threshold', 'narrow_eps_threshold'])
def test_cubic_round_trip_and_log_derivative_vs_autograd(opt):
    K = 16
    opts = _cub_opts(opt, K)
    uw, uh, ud = _dev(*_params(K, 2, seed=13))
    x = _inputs(LO, HI, seed=14).to(DEV).requires_grad_(True)
    y, ld = CUB(x, uw, uh, ud, lower=LO, upper=HI, **opts)
    xr, ldr = CUB(y.detach(), uw, uh, ud, inverse=True, lower=LO, upper=HI, **opts)
    # the reference's own cubic round trip has outliers of this frequency (see test_gpu_parity.py)
    assert ((xr - x.detach()).abs() > 1e-4).float().mean().item() <= 2e-3
    assert ((ldr + ld.detach()).abs() > 1e-4).float().mean().item() <= 2e-3
    dydx, = torch.autograd.grad(y.sum(), x)
    torch.testing.assert_close(dydx.log(), ld.detach(), rtol=0, atol=1e-4)


def _reference_checkers():
    """tests/golden/ref_tests/base.py -- the reference's own checkers, unchanged -- imported with `stribor`
    resolving to this package, as tests/golden/ref_tests/conftest.py does."""
    if 'stribor.test.base' in sys.modules:
        return sys.modules['stribor.test.base']
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
    stubs = os.path.join(golden, '_stubs')
    if stubs not in sys.path:
        sys.path.append(stubs)              # annotation-only `torchtyping`
    sys.modules.setdefault('stribor', st)
    spec = importlib.util.spec_from_file_location('spline_options_ref_base', os.path.join(golden, 'ref_tests', 'base.py'))
    base = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(base)
    return base


class MinDerivativeSpline(st.Spline):
    """The reference's subclassing pattern (ref_tests/test_spline.py: UnboundedSpline) with a spline option."""

    def forward_and_log_diag_jacobian(self, x, latent=None, *, reverse=False, **kwargs):
        w, h, d = self._get_params(latent)
        return self.spline(x, w, h, d, inverse=reverse, lower=self.lower, upper=self.upper, min_derivative=1e-4)


@gpu
@pytest.mark.parametrize('input_shape', [(1, 1), (2, 10), (10, 2), (7, 4, 5)])
def test_spline_subclass_with_option_passes_reference_checkers(input_shape):
    base = _reference_checkers()
    torch.manual_seed(123)
    torch.set_default_device(DEV)
    try:
        x = torch.rand(*input_shape) * 2
        f = MinDerivativeSpline(dim=input_shape[-1], n_bins=5, lower=0, upper=2, spline_type='quadratic')
        base.check_inverse_transform(f, x)
        base.check_log_jacobian_determinant(f, x)
        base.check_gradients_not_nan(f, x)
    finally:
        torch.set_default_device('cpu')


# ------------------------------------------------------------------------------------------------------------
# errors
# ------------------------------------------------------------------------------------------------------------
@gpu
def test_option_errors():
    K = 16
    x = _inputs(LO, HI, seed=15).to(DEV)
    uw, uh, ud = _dev(*_params(K, K - 1, seed=16))
    with pytest.raises(ValueError, match='bin width'):
        RQS(x, uw, uh, ud, min_bin_width=0.07)
    with pytest.raises(ValueError, match='bin height'):
        RQS(x, uw, uh, ud, min_bin_height=0.07)
    with pytest.raises(ValueError, match='bin width'):
        CUB(x, uw, uh, ud[..., :2], min_bin_width=0.07)
    with pytest.raises(ValueError, match='bin height'):
        CUB(x, uw, uh, ud[..., :2], min_bin_height=0.07)
    with pytest.raises(ValueError):
        RQS(x, uw, uh, ud, min_derivative=-1e-3)
    with pytest.raises(ValueError):
        RQS(x, uw, uh, ud, min_derivative=float('nan'))
    with pytest.raises(ValueError):
        CUB(x, uw, uh, ud[..., :2], eps=float('inf'))
    for n_der in (K, K - 2, K + 2):
        with pytest.raises(ValueError, match='entries'):
            RQS(x, uw, uh, _dev(_params(K, n_der, seed=17)[2])[0])
    t = torch.tensor(1., device=DEV)
    with pytest.raises(NotImplementedError):
        RQS(x, uw, uh, ud, left=-t, right=t, bottom=-t, top=t, min_derivative=1e-2)
    # min * K == 1 is allowed (every bin has the same size)
    RQS(x, uw, uh, ud, min_bin_width=1 / K, min_bin_height=1 / K)


# ------------------------------------------------------------------------------------------------------------
# host side: the C ABI (no GPU needed)
# ------------------------------------------------------------------------------------------------------------
def _coupling_struct(fmeta, dim=64, n_bins=16, kind=_lib.RQS):
    """stb_layer of Coupling(Spline(dim, 16), MLP(dim, [64], dim * P)): a layer the tensor-core kernels take.
    The weight pointers are CPU tensors; the host-side entry points never dereference them."""
    hidden = 64
    P = 3 * n_bins - 1 if kind == _lib.RQS else 2 * n_bins + 2
    mask_list = [0] * (dim // 2) + [1] * (dim - dim // 2)
    meta = [kind, dim, 0, 1, 0, n_bins, 0, 0, _lib.ACTIVATIONS['Tanh'], 0, 2, 4, 0, 0, dim, hidden, dim * P] + mask_list
    params = [torch.zeros(hidden, dim), torch.zeros(hidden), torch.zeros(dim * P, hidden), torch.zeros(dim * P)]
    mask = torch.tensor(mask_list, dtype=torch.uint8)
    L = _ops.make_struct(meta, fmeta, mask, params, None)
    L._keep = (params, mask)
    return L


def test_fmeta_without_options_means_defaults():
    L = _coupling_struct([-4., 4., 0., 1., 0., 1.])
    assert L.spline.custom == 0 and L.spline.free_edge_derivs == 0 and L.spline.min_derivative == 0.0
    L = _coupling_struct([-4., 4., 0., 1., 0., 1., 1., 2e-2, 1e-4, 0.1, 1., 1e-6, 1e-4])
    o = L.spline
    assert (o.custom, o.free_edge_derivs) == (1, 1)
    assert [o.min_bin_width, o.min_bin_height, o.min_derivative, o.cub_eps, o.cub_quad_threshold] == \
        [float(np.float32(v)) for v in (2e-2, 1e-4, 0.1, 1e-6, 1e-4)]
    assert C.sizeof(_lib.StbLayer) == _lib.lib().stb_sizeof_layer()


@pytest.mark.parametrize('kind', [_lib.RQS, _lib.CUBIC])
@pytest.mark.parametrize('dim', [64, 128])
def test_custom_options_never_take_a_tensor_core_path(kind, dim):
    lib = _lib.lib()
    plain = _coupling_struct([-4., 4., 0., 1., 0., 1.], dim=dim, kind=kind)
    assert lib.stb_packed_bytes(C.byref(plain)) > 0
    custom = _coupling_struct([-4., 4., 0., 1., 0., 1., 1., 1e-3, 1e-3, 1e-3, 0., 1e-5, 1e-3], dim=dim, kind=kind)
    assert lib.stb_packed_bytes(C.byref(custom)) == 0
    custom.packed = 1                             # a packed image would not be used either
    assert lib.stb_layer_uses_tensor_path(C.byref(custom)) == 0
    # the wide-conditioner family (MLP[128])
    wide = _coupling_struct([-4., 4., 0., 1., 0., 1.], dim=32, kind=kind)
    wide.net.dims[1] = 128
    assert lib.stb_packed_bytes(C.byref(wide)) > 0
    wide.spline.custom = 1
    wide.spline.min_bin_width = wide.spline.min_bin_height = 1e-2
    assert lib.stb_packed_bytes(C.byref(wide)) == 0


def test_option_validation_in_the_c_abi():
    lib = _lib.lib()

    def ok(**kw):
        L = _coupling_struct([-4., 4., 0., 1., 0., 1.], dim=8)
        L.net.dims[2] = 8 * (3 * 16 + 1 if kw.get('free_edge_derivs') else 3 * 16 - 1)
        L.spline.custom = 1
        for k, v in {'min_bin_width': 1e-3, 'min_bin_height': 1e-3, 'min_derivative': 1e-3, **kw}.items():
            setattr(L.spline, k, v)
        # validates the layer first (E_INVAL), then refuses a layer with a network (E_NOTSUP) before any launch
        return lib.stb_layer_backward_diag(C.byref(L), _lib.FORWARD, None, None, None, None, None, 0, None)

    assert ok() == _lib.E_NOTSUP
    assert ok(free_edge_derivs=1) == _lib.E_NOTSUP
    assert ok(min_bin_width=1 / 16, min_bin_height=1 / 16) == _lib.E_NOTSUP
    assert ok(min_bin_width=0.07) == _lib.E_INVAL
    assert ok(min_bin_height=0.07) == _lib.E_INVAL
    assert ok(min_derivative=-1e-3) == _lib.E_INVAL
    assert ok(min_derivative=float('inf')) == _lib.E_INVAL
