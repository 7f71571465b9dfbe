"""CPU: host-side logic -- masks, state-dict compatibility, descriptors, the C ABI surface."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import cases
from golden_util import blob
import stribor_b200 as st
from stribor_b200 import _lib, _ops
from stribor_b200.spec import layers_from_spec, spec_from_layers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_masks_match_reference_vectors():
    for k, v in blob().items():
        if k.startswith('mask|'):
            _, nm, d = k.split('|')
            assert np.array_equal(st.util.get_mask(nm)(int(d)).numpy(), v), k
    with pytest.raises(NotImplementedError):
        st.util.get_mask('nope')
    g = st.util.get_mask('random_half')
    assert torch.equal(g(10), g(10)) and g(10).sum() == 5      # frozen after the first draw
    assert torch.equal(g(1), torch.ones(1))


def test_state_dict_keys_match_reference_layout():
    d = 4
    f = st.NormalizingFlow(st.UnitNormal(d), [
        st.Coupling(st.Spline(d, 8, latent_net=st.net.MLP(d, [16, 16], d * 23), spline_type='quadratic'),
                    mask='ordered_right_half'),
        st.Coupling(st.Affine(d, latent_net=st.net.MLP(d, [16], 2 * d)), mask='ordered_left_half'),
        st.ContinuousAffineCoupling(st.net.MLP(d + 1, [8], 2 * d), st.net.TimeLinear(2 * d), 'parity_odd'),
        st.Affine(d), st.Spline(d, 3)])
    keys = list(f.state_dict().keys())
    assert keys == [
        'transforms.0.transform.latent_net.net.0.weight', 'transforms.0.transform.latent_net.net.0.bias',
        'transforms.0.transform.latent_net.net.2.weight', 'transforms.0.transform.latent_net.net.2.bias',
        'transforms.0.transform.latent_net.net.4.weight', 'transforms.0.transform.latent_net.net.4.bias',
        'transforms.1.transform.latent_net.net.0.weight', 'transforms.1.transform.latent_net.net.0.bias',
        'transforms.1.transform.latent_net.net.2.weight', 'transforms.1.transform.latent_net.net.2.bias',
        'transforms.2.latent_net.net.0.weight', 'transforms.2.latent_net.net.0.bias',
        'transforms.2.latent_net.net.2.weight', 'transforms.2.latent_net.net.2.bias',
        'transforms.2.time_net.scale',
        'transforms.3.log_scale', 'transforms.3.shift',
        'transforms.4.width', 'transforms.4.height', 'transforms.4.derivative']
    # last Linear bias is zero-initialised (mlp.py:53)
    assert float(f.transforms[0].transform.latent_net.net[4].bias.abs().sum()) == 0.0
    # fixed-scale Affine holds no state (affine.py:50-57)
    assert list(st.Affine(2, scale=2., shift=1.).state_dict().keys()) == []
    with pytest.raises(AssertionError):
        st.Affine(2, scale=-1., shift=0.)


def test_descriptor_wire_format():
    d = 6
    c = st.Coupling(st.Spline(d, 5, latent_net=st.net.MLP(d + 3, [7, 9], d * 14), lower=-2, upper=3,
                              spline_type='quadratic'), mask='parity_even')
    desc = c.describe(d, 3, 'cpu')
    m = desc['meta']
    assert m[:_ops.META_HEADER] == [_lib.RQS, d, 3, 1, 0, 5, 0, 0, _lib.ACTIVATIONS['Tanh'], 0, 3, 6, 0, 0]
    assert m[_ops.META_HEADER:] == [d + 3, 7, 9, d * 14] + [0, 1, 0, 1, 0, 1]
    assert _ops.meta_len(m) == len(m)
    assert desc['fmeta'][:2] == [-2.0, 3.0]
    assert desc['mask'].tolist() == [0, 1, 0, 1, 0, 1] and desc['mask'].dtype == torch.uint8
    assert [tuple(p.shape) for p in desc['params']] == [(7, 9), (7,), (9, 7), (9,), (84, 9), (84,)]
    L = _ops.make_struct(desc['meta'], desc['fmeta'], desc['mask'], desc['params'])
    assert (L.kind, L.dim, L.latent_dim, L.cond_x, L.n_bins, L.net.n_linear) == (_lib.RQS, d, 3, 1, 5, 3)
    assert list(L.net.dims)[:4] == [9, 7, 9, 84]
    assert L.net.W[2] == desc['params'][4].data_ptr() and L.mask == desc['mask'].data_ptr()
    assert list((ctypes.c_uint8 * d).from_address(L.mask_host)) == [0, 1, 0, 1, 0, 1]
    # d == 1 -> conditioning zeroed (coupling.py:62-63); 'none' mask -> everything transformed
    c1 = st.Coupling(st.Affine(1, latent_net=st.net.MLP(1, [4], 2)), mask='none')
    d1 = c1.describe(1, 0, 'cpu')
    assert d1['meta'][7] == 1 and d1['mask'].tolist() == [0]
    # continuous affine: time is the last network input, TimeLinear(2) broadcasts (README.md:94-97)
    ca = st.ContinuousAffineCoupling(st.net.MLP(4 + 1, [8], 8), st.net.TimeLinear(2), 'ordered_0')
    dc = ca.describe(4, 0, 'cpu')
    assert dc['meta'][0] == _lib.CONT_AFFINE and dc['meta'][4] == 1 and dc['params'][-1].shape == (8,)
    s = ca.time_net.scale.detach().view(-1)
    assert torch.equal(dc['params'][-1].detach(), torch.stack([s[0]] * 4 + [s[1]] * 4))
    # conditioners the kernels cannot fuse are not describable (they run as modules around the
    # element-wise kernels instead, see test_gpu_parity.py::test_foreign_conditioner)
    with pytest.raises(NotImplementedError):
        st.Coupling(st.Affine(2, latent_net=torch.nn.Linear(2, 4)), mask='ordered_0').describe(2, 0, 'cpu')
    with pytest.raises(NotImplementedError):
        st.Coupling(st.Affine(2, latent_net=st.net.MLP(2, [4], 4, activation='Hardtanh')),
                    mask='ordered_0').describe(2, 0, 'cpu')


@pytest.mark.parametrize('name', ['quadratic_d5_parity', 'cubic_d7_ordered', 'neural_flow_d16_L4',
                                  'affine_coupling_2x10_l13', 'spline_cubic_7x4x5_k3_l0'])
def test_spec_roundtrip(name):
    spec = cases.build_case(name)['spec']
    back = spec_from_layers(layers_from_spec(spec))

    def flat(v):
        if isinstance(v, torch.Tensor):
            return [v]
        if isinstance(v, dict):
            return [t for k in sorted(v) for t in flat(v[k])]
        if isinstance(v, (list, tuple)):
            return [t for u in v for t in flat(u)]
        return []
    a, b = flat(spec), flat(back)
    assert len(a) == len(b) and all(torch.equal(x, y) for x, y in zip(a, b))
    assert [l['type'] for l in spec] == [l['type'] for l in back]


def test_cpu_tensors_are_refused_not_emulated():
    f = st.Coupling(st.Affine(4, latent_net=st.net.MLP(4, [8], 8)), mask='ordered_0')
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        f(torch.randn(3, 4))
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        st.NormalizingFlow(st.UnitNormal(4), [f]).log_prob(torch.randn(3, 4))


def test_cabi_library_loads_and_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, 'include', 'stribor_b200.h')).read()
    declared = set(re.findall(r'\b(stb_[a-z_0-9]+)\s*\(', header))
    declared -= {'stb_layer', 'stb_mlp'}
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    l = _lib.lib()
    for name in declared:
        assert hasattr(l, name), name
    assert l.stb_abi_version() == _lib.ABI_VERSION
    assert l.stb_sizeof_layer() == ctypes.sizeof(_lib.StbLayer)
    assert isinstance(l.stb_last_error(), bytes)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, 'stribor_b200')
    for dp, _, fs in os.walk(pkg):
        for fn in fs:
            if fn.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dp, fn)).read()
                assert 'import oracle' not in src and 'from oracle' not in src, fn


def test_backward_workspace_layout_constants_match_the_kernels():
    """The Python side un-packs the fused backward's workspace (stribor_b200/_ops.py); its layout constants and the
    packed column order must match tc_wide.cu (read from the source: no GPU needed)."""
    import re
    from stribor_b200 import _ops
    src = open(os.path.join(ROOT, 'stribor_b200', 'csrc', 'tc_wide.cu')).read()

    def const(name):
        m = re.search(r'constexpr\s+int\s+' + name + r'\s*=\s*(\d+)\s*;', src)
        assert m, name
        return int(m.group(1))

    assert _ops.G_PAD == const('kPPad') == 48
    assert _ops.H_AUG == const('kHAug') == const('kWStride') == 72
    # natural parameter p -> packed column (w_i, h_i interleaved, then the derivative columns): inverse of
    # param_of_col() in the pack kernels
    cols = _ops._packed_cols(torch.device('cpu')).tolist()
    bins = 16

    def param_of_col(c):
        return (bins + (c >> 1) if (c & 1) else (c >> 1)) if c < 2 * bins else c

    assert sorted(cols) == list(range(48))
    assert all(param_of_col(c) == p for p, c in enumerate(cols))


def _spline_struct(dim, kind='quadratic', hidden=64, n_bins=16, latent_dim=0, act='Tanh', time_input=0, inv_own=0,
                   custom=0, mask=None):
    """stb_layer for Coupling(Spline(dim, n_bins), MLP(dim, [hidden], dim * P)) with an ordered mask (kind 'affine' /
    'cont': Affine / ContinuousAffineCoupling, hidden may be a list); the weight pointers are CPU tensors -- the
    host-side entry points below never dereference them."""
    from stribor_b200 import _lib, _ops
    kinds = {'quadratic': _lib.RQS, 'cubic': _lib.CUBIC, 'affine': _lib.AFFINE, 'cont': _lib.CONT_AFFINE}
    P = {'quadratic': 3 * n_bins - 1, 'cubic': 2 * n_bins + 2}.get(kind, 2)
    hidden = list(hidden) if isinstance(hidden, (list, tuple)) else [hidden]
    dims = [dim + latent_dim + time_input] + hidden + [dim * P]
    mask_list = mask if mask is not None else [0] * (dim // 2) + [1] * (dim - dim // 2)
    params = []
    for i in range(len(dims) - 1):
        params += [torch.zeros(dims[i + 1], dims[i]), torch.zeros(dims[i + 1])]
    if kind == 'cont':
        params.append(torch.zeros(2 * dim))                    # TimeLinear.scale
    meta = [kinds[kind], dim, latent_dim, 1, time_input, n_bins, inv_own, 0, _lib.ACTIVATIONS[act], 0,
            len(dims) - 1, len(params), 0, 0] + dims + mask_list
    fmeta = [-4., 4., 0., 1., 0., 1.] + ([1, 1e-2, 1e-2, 1e-2, 0, 1e-6, 1e-3] if custom else [])
    mask = torch.tensor(mask_list, dtype=torch.uint8)
    L = _ops.make_struct(meta, fmeta, mask, params, None)
    L._keep = (params, mask)
    return L


def test_cabi_host_side_dispatch_without_a_gpu():
    """Which layers get which tensor-core images / the fused backward, and argument validation: host logic of the
    C ABI (no kernel is launched, no device pointer is touched)."""
    import ctypes as C
    from stribor_b200 import _lib
    lib = _lib.lib()
    tc_bytes = 8192 + 12288 + 16 * 24576                       # tc_layer.cu image (dim <= 64)
    wide_bytes = 16384 + 24576 + 32 * 24576                    # tc_wide.cu image (dim <= 128)
    ws = lambda rows: 4 * (rows * 72 + 64 * 48 * 72 + 64 * 64 + 64)
    for kind in ('quadratic', 'cubic'):
        L64, L128, L130 = _spline_struct(64, kind), _spline_struct(128, kind), _spline_struct(130, kind)
        assert lib.stb_packed_bytes(C.byref(L64)) == tc_bytes + wide_bytes      # both images: 256-row inference + 128-row / backward
        assert lib.stb_packed_bytes(C.byref(L128)) == wide_bytes
        assert lib.stb_packed_bytes(C.byref(L130)) == 0                          # 65 transformed dims: CUDA-core kernel only
        assert lib.stb_layer_backward_workspace_bytes(C.byref(L128), 1000) == ws(1000)
        assert lib.stb_layer_backward_workspace_bytes(C.byref(L64), 7) == ws(7)
        assert lib.stb_layer_backward_workspace_bytes(C.byref(L130), 1000) == 0
    assert lib.stb_packed_bytes(C.byref(_spline_struct(64, hidden=32))) == 0     # MLP[32]: no tensor-core path
    assert lib.stb_layer_backward_workspace_bytes(C.byref(_spline_struct(64, n_bins=8)), 10) == 0
    # round 2: 2..15 bins and `latent=` inputs keep the tensor-core FORWARD images (the fused backward needs 16 bins, no latent)
    assert lib.stb_packed_bytes(C.byref(_spline_struct(64, n_bins=8))) == tc_bytes + wide_bytes
    assert lib.stb_packed_bytes(C.byref(_spline_struct(128, n_bins=5, kind='cubic'))) == wide_bytes
    assert lib.stb_packed_bytes(C.byref(_spline_struct(64, n_bins=1))) == 0
    assert lib.stb_packed_bytes(C.byref(_spline_struct(64, n_bins=17))) == 0
    assert lib.stb_packed_bytes(C.byref(_spline_struct(32, latent_dim=8))) == tc_bytes + wide_bytes     # 16 + 8 <= 32 K columns
    assert lib.stb_packed_bytes(C.byref(_spline_struct(64, latent_dim=16))) == wide_bytes               # 32 + 16 > 32: 128-row kernel
    assert lib.stb_packed_bytes(C.byref(_spline_struct(64, latent_dim=40))) == 0                        # 32 + 40 > 64
    assert lib.stb_layer_backward_workspace_bytes(C.byref(_spline_struct(32, latent_dim=8)), 10) == 0
    big = lib.stb_packed_bytes(C.byref(_spline_struct(64, hidden=256, n_bins=10)))                      # wide conditioner, MLP[256]
    assert big > tc_bytes and lib.stb_packed_bytes(C.byref(_spline_struct(64, hidden=256, n_bins=16))) == big
    # wide-conditioner splines (tc_hwide.cu): header + biases 9216 B, W1 6 blocks of [H x 16] bf16, W2 (H / 16) blocks of
    # [H x 16] hi | lo, W3 32 dims x [48 x H] hi | lo
    hw = lambda H, n_hidden: 9216 + 6 * H * 32 + (H // 16 * H * 64 if n_hidden == 2 else 0) + 32 * H * 192
    assert big == hw(256, 1)
    assert lib.stb_packed_bytes(C.byref(_spline_struct(64, hidden=[64, 64]))) == hw(64, 2)
    assert lib.stb_packed_bytes(C.byref(_spline_struct(64, hidden=128, kind='cubic'))) == hw(128, 1)
    # affine / continuous-affine (tc_mlp.cu): 4096 B header + biases, W1 6 blocks, W2 (H / 16) blocks, W3 (H / 16) x [64 x 16]
    mlp = lambda H, n_hidden: 4096 + 6 * H * 32 + (H // 16 * H * 64 if n_hidden == 2 else 0) + H // 16 * 4096
    assert lib.stb_packed_bytes(C.byref(_spline_struct(32, kind='affine'))) == mlp(64, 1)
    assert lib.stb_packed_bytes(C.byref(_spline_struct(64, kind='affine', hidden=[256, 256]))) == mlp(256, 2)
    assert lib.stb_packed_bytes(C.byref(_spline_struct(16, kind='cont', time_input=1))) == mlp(64, 1)
    # no tensor-core path: H = 96, an unbounded activation, conditioning + t + latent over GEMM1's 32 columns, custom
    # spline constants, the layer's own inverse log-det
    for L in (_spline_struct(64, hidden=96), _spline_struct(64, kind='affine', hidden=96), _spline_struct(64, act='ReLU'),
              _spline_struct(32, kind='affine', act='ReLU'), _spline_struct(64, kind='cont', time_input=1, latent_dim=0),
              _spline_struct(32, kind='cont', time_input=1, latent_dim=16), _spline_struct(64, custom=1),
              _spline_struct(64, hidden=256, custom=1), _spline_struct(64, inv_own=1), _spline_struct(32, kind='affine', inv_own=1)):
        assert lib.stb_packed_bytes(C.byref(L)) == 0
        assert lib.stb_layer_uses_tensor_path(C.byref(L)) == 0
    # log_prob without the [rows, dim] scratch: two packed layers of each chain family go out as one launch
    for a, b in ((_spline_struct(64), _spline_struct(64, mask=[1] * 32 + [0] * 32)),
                 (_spline_struct(16, kind='affine'), _spline_struct(16, kind='affine')),
                 (_spline_struct(16, kind='cont', time_input=1), _spline_struct(16, kind='cont', time_input=1))):
        for L in (a, b):
            L.packed, L.packed_bytes = 0x1000, lib.stb_packed_bytes(C.byref(L))
            assert lib.stb_layer_uses_tensor_path(C.byref(L)) == 1
        assert lib.stb_flow_log_prob_needs_x_out((_lib.StbLayer * 2)(a, b), 2) == 0
    # argument validation returns STB_EINVAL (-1) before anything is launched
    L = _spline_struct(64)
    dummy = C.c_void_p(0x1000)
    assert lib.stb_flow_apply(C.byref(L), 0, 0, dummy, None, None, dummy, None, 0, 10, None) == _lib.E_INVAL
    assert b'empty flow' in lib.stb_last_error()
    assert lib.stb_layer_apply(C.byref(L), 7, dummy, None, None, dummy, None, 0, 0, 10, None) == _lib.E_INVAL
    assert lib.stb_flow_log_prob(C.byref(L), 1, dummy, None, None, None, None, 10, None) == _lib.E_INVAL
    # rows == 0 is a no-op that touches nothing
    assert lib.stb_layer_apply(C.byref(L), 0, dummy, None, None, dummy, None, 0, 0, 0, None) == 0
    assert lib.stb_flow_log_prob(C.byref(L), 1, dummy, None, None, dummy, dummy, 0, None) == 0


def test_call_plan_records_follow_structure_and_parameter_changes():
    """flow.run_chain's cache bookkeeping (no GPU needed): a record per ModuleList, rebuilt when the structure epoch
    moves (attribute set on one of this package's modules, parameter / sub-module registered anywhere, packed image
    dropped), its plans dropped when a parameter's (data_ptr, _version, requires_grad) changes; weak keys."""
    import copy
    import gc
    import weakref
    import stribor_b200 as st
    from stribor_b200 import _epoch, flow as F

    def make():
        return st.NormalizingFlow(st.UnitNormal(8), [
            st.Coupling(st.Spline(8, 4, latent_net=st.net.MLP(8, [16], 8 * 11), lower=-3, upper=3, spline_type='quadratic'),
                        mask=m) for m in ('ordered_right_half', 'ordered_left_half')])

    flow = make()
    rec = F._record(flow.transforms)
    assert rec.chainable and len(rec.plist) == 8 and rec.any_grad
    assert F._record(flow.transforms) is rec                       # nothing moved
    rec.plans['sentinel'] = object()
    # in-place parameter update: same record, plans dropped
    lin = [m for m in flow.modules() if isinstance(m, torch.nn.Linear)]
    with torch.no_grad():
        lin[0].weight.mul_(2.0)
    assert F._record(flow.transforms) is rec and not rec.plans
    rec.plans['sentinel'] = object()
    lin[1].bias.requires_grad_(False)                              # requires_grad is part of the token
    assert F._record(flow.transforms) is rec and not rec.plans
    # attribute of one of this package's modules
    e0 = _epoch.value
    flow.transforms[0].transform.lower = -5.0
    assert _epoch.value > e0 and F._record(flow.transforms) is not rec
    rec = F._record(flow.transforms)
    # a parameter object replaced, a sub-module appended, a packed image dropped: all move the epoch
    for change in (lambda: setattr(lin[0], 'bias', torch.nn.Parameter(torch.zeros_like(lin[0].bias))),
                   lambda: flow.transforms.append(make().transforms[0]),
                   lambda: st.invalidate_packed(flow)):
        e0 = _epoch.value
        change()
        assert _epoch.value > e0
        new = F._record(flow.transforms)
        assert new is not rec
        rec = new
    assert len(rec.plist) == 12
    # gradients off / on decide the fused path, per call
    with torch.no_grad():
        assert F._chain_ok(flow.transforms, (None,))
    assert not F._chain_ok(flow.transforms, (None,))              # parameters require grad
    flow.requires_grad_(False)
    assert F._chain_ok(flow.transforms, (None,))
    assert not F._chain_ok(flow.transforms, (torch.zeros(1, requires_grad=True),))
    # foreign modules never chain; records do not keep flows alive; flows stay deep-copyable
    foreign = st.NormalizingFlow(st.UnitNormal(8), [torch.nn.Identity()])
    assert not F._chain_ok(foreign.transforms, (None,))
    copy.deepcopy(flow)
    ref = weakref.ref(flow.transforms)
    del flow, rec, new, lin, change
    gc.collect()
    assert ref() is None


@pytest.mark.parametrize('name', ['TimeIdentity', 'TimeLinear', 'TimeTanh', 'TimeLog', 'TimeFourier', 'TimeFourierBounded'])
def test_time_embeddings_vanish_at_zero_and_match_their_derivative(name):
    """The reference's time embeddings (net/time_net.py): phi(0) = 0, `derivative` is d phi / dt, shapes [..., out]."""
    import stribor_b200 as st
    torch.manual_seed(3)
    cls = getattr(st.net, name)
    net = cls(6, hidden_dim=5) if 'Fourier' in name else cls(6)
    t = torch.rand(4, 3, 1, dtype=torch.float64) * 2
    net = net.double()
    assert net(torch.zeros(4, 3, 1, dtype=torch.float64)).abs().max() == 0
    out = net(t)
    assert out.shape == (4, 3, 6)
    tg = t.clone().requires_grad_(True)
    want = torch.stack([torch.autograd.grad(net(tg)[..., j].sum(), tg, retain_graph=True)[0][..., 0] for j in range(6)], -1)
    torch.testing.assert_close(net.derivative(t).expand_as(want), want, rtol=1e-10, atol=1e-12)
    if name == 'TimeFourierBounded':
        assert out.abs().max() <= 0.5


def test_subclasses_that_override_behaviour_are_not_fused():
    """The fused kernels stand in for a module only when it IS the class they implement: a subclass that overrides
    forward (the reference derives TimeTanh / TimeLog from TimeLinear exactly like that) must run as the module it is."""
    import stribor_b200 as st
    from stribor_b200.flows._native import fusable

    class Doubled(st.net.MLP):
        def forward(self, x):
            return 2 * super().forward(x)

    class MyTime(st.net.TimeLinear):
        def forward(self, t):
            return torch.sin(self.scale * t)

    class Clamped(st.Affine):
        def forward(self, x, latent=None, **kw):
            return super().forward(x.clamp(-1, 1), latent=latent, **kw)

    assert fusable(st.net.MLP(4, [8], 8)) and not fusable(Doubled(4, [8], 8))
    mk = lambda tn: st.ContinuousAffineCoupling(st.net.MLP(5, [8], 8), tn, 'ordered_0')
    assert mk(st.net.TimeLinear(8)).chainable()
    for tn in (MyTime(8), st.net.TimeTanh(8), st.net.TimeLog(8), st.net.TimeIdentity(8)):
        assert not mk(tn).chainable(), type(tn).__name__
    assert st.Coupling(st.Affine(4, latent_net=st.net.MLP(4, [8], 8)), 'ordered_0').chainable()
    assert not st.Coupling(st.Affine(4, latent_net=Doubled(4, [8], 8)), 'ordered_0').chainable()
    assert not st.Coupling(Clamped(4, latent_net=st.net.MLP(4, [8], 8)), 'ordered_0').chainable()
    assert st.Affine(4, latent_net=st.net.MLP(3, [8], 8)).plain() and not Clamped(4, latent_net=st.net.MLP(3, [8], 8)).plain()


def test_layer_subclasses_that_override_the_transform_methods_leave_the_fused_chain():
    import stribor_b200 as st
    from stribor_b200 import flow as F

    class Noisy(st.Coupling):
        def forward(self, x, **kw):
            return super().forward(x + 1.0, **kw)

    class Same(st.Coupling):                      # adds state, overrides nothing the kernels replace
        def extra(self):
            return 1

    mk = lambda cls: cls(st.Affine(4, latent_net=st.net.MLP(4, [8], 8)), 'ordered_0')
    assert mk(st.Coupling).chainable() and mk(Same).chainable() and not mk(Noisy).chainable()
    assert st.Flip().chainable()

    class MyFlip(st.Flip):
        def inverse(self, y, **kw):
            return y
    assert not MyFlip().chainable()
    flow = st.NormalizingFlow(st.UnitNormal(4), [mk(st.Coupling), mk(Noisy)]).requires_grad_(False)
    assert not F._chain_ok(flow.transforms, (None,))
