"""Generate tests/golden/reference_outputs.npz by running the UNMODIFIED reference.

Run in the build container only (the reference does not travel to the GPU box):

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

The reference (/root/reference, stribor 0.2.0) imports two packages this image lacks;
``tests/golden/_stubs`` holds annotation-only stand-ins (SURVEY.md section 8c).  For every
case in ``cases.py`` the reference modules are built, their parameters overwritten with the
portable numpy-generated weights, and the listed ops evaluated in fp32 and in fp64.
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

# An array of more than LARGE elements (the NLL gradients of the wide last Linear layers) is stored as a fixed sample
# of SAMPLE_ROWS of its rows, their indices under 'case|key|rows'; the tests compare those rows.
LARGE = 1 << 16
SAMPLE_ROWS = 256


def sample_large(blob):
    for k in [k for k, v in blob.items() if v.size > LARGE]:
        case, key, _ = k.split('|')
        rows = np.sort(np.random.RandomState(0).choice(blob[k].shape[0], SAMPLE_ROWS, replace=False))
        blob[k] = blob[k][rows]
        blob[f'{case}|{key}|rows'] = rows
    return blob


def _load_mlp(ref_mlp, net):
    lin = [m for m in ref_mlp.net if isinstance(m, torch.nn.Linear)]
    assert len(lin) == len(net['weights'])
    for m, w, b in zip(lin, net['weights'], net['biases']):
        assert m.weight.shape == w.shape, (m.weight.shape, w.shape)
        m.weight.data = w.clone()
        m.bias.data = b.clone()


def _dims(net):
    ws = net['weights']
    return ws[0].shape[1], [w.shape[0] for w in ws[:-1]], ws[-1].shape[0]


def _ref_mlp(net):
    i, h, o = _dims(net)
    m = st.net.MLP(i, h, o, activation=net['activation'], final_activation=net['final_activation'])
    _load_mlp(m, net)
    return m


def _ref_transform(tr):
    net = _ref_mlp(tr['net']) if tr.get('net') is not None else None
    if tr['kind'] == 'affine':
        f = st.Affine(tr['dim'], latent_net=net)
        if net is None:
            f.log_scale.data, f.shift.data = tr['params'][0].clone(), tr['params'][1].clone()
        return f
    f = st.Spline(tr['dim'], tr['n_bins'], latent_net=net, lower=tr['lower'], upper=tr['upper'],
                  spline_type=tr['kind'])
    if net is None:
        f.width.data, f.height.data, f.derivative.data = [p.clone() for p in tr['params']]
    return f


def ref_layer(layer):
    if layer['type'] == 'sigmoid':
        return st.Sigmoid()
    if layer['type'] == 'logit':
        return st.Logit()
    if layer['type'] == 'flip':
        return st.Flip()
    if layer['type'] == 'permute':
        f = st.Permute(len(layer['perm']))
        f.permutation = torch.as_tensor(layer['perm']).long()
        f.inverse_permutation = torch.empty_like(f.permutation)
        f.inverse_permutation[f.permutation] = torch.arange(len(layer['perm']))
        return f
    if layer['type'] == 'elementwise':
        return _ref_transform(layer['transform'])
    if layer['type'] == 'coupling':
        return st.Coupling(_ref_transform(layer['transform']), mask=layer['mask'])
    if layer['type'] == 'cont_affine_coupling':
        tn = st.net.TimeLinear(layer['time_scale'].shape[-1])
        tn.scale.data = layer['time_scale'].clone()
        return st.ContinuousAffineCoupling(_ref_mlp(layer['net']), tn, layer['mask'],
                                           concatenate_time=layer['concatenate_time'])
    raise ValueError(layer['type'])


def run_case(name, dtype):
    torch.set_default_dtype(dtype)
    case = cases.build_case(name)
    layers = [ref_layer(l) for l in case['spec']]
    for l in layers:
        l.to(dtype)
    inp = {k: v.to(dtype) for k, v in case['inputs'].items()}
    x = inp['x']
    kw = {k: inp[k] for k in ('latent', 't') if k in inp}
    dim = x.shape[-1]
    out = {}
    flow = st.NormalizingFlow(st.UnitNormal(dim), layers)
    capture = []
    orig_ss = st.util.searchsorted

    def spy(knots, v, eps=1e-6):
        r = orig_ss(knots, v, eps)
        capture.append(r.detach().clone())
        return r

    for op in case['ops']:
        if op == 'forward_ldj':
            with torch.no_grad():
                st.util.searchsorted = spy
                capture.clear()
                y, ldj = flow.forward_and_log_det_jacobian(x, **kw)
                st.util.searchsorted = orig_ss
            out['forward.y'], out['forward.ldj'] = y, ldj
            if name.startswith('spline_') and len(capture) == 1:
                out['forward.bins'] = capture[0]
        elif op == 'inverse_ldj':
            with torch.no_grad():
                st.util.searchsorted = spy
                capture.clear()
                xr, ldj = flow.inverse_and_log_det_jacobian(x, **kw)
                st.util.searchsorted = orig_ss
            out['inverse.x'], out['inverse.ldj'] = xr, ldj
            if name.startswith('spline_') and len(capture) == 1:
                out['inverse.bins'] = capture[0]
        elif op == 'inverse_ldj_unit':       # inverse of a flow that ends in (0, 1): feed the forward output
            with torch.no_grad():
                y = flow.forward(x, **kw)
                xr, ldj = flow.inverse_and_log_det_jacobian(y, **kw)
            out['inverse_unit.y'], out['inverse_unit.x'], out['inverse_unit.ldj'] = y, xr, ldj
        elif op == 'log_prob':
            with torch.no_grad():
                out['log_prob'] = flow.log_prob(x, **kw)
        elif op in ('neural_flow', 'neural_flow_t0'):
            nf = st.NeuralFlow(layers)
            with torch.no_grad():
                if op == 'neural_flow':
                    out['neural_flow.y'] = nf(x, t=inp['t'])
                else:
                    out['neural_flow_t0.y'] = nf(x, t=inp['t'], t0=inp['t0'])
        elif op == 'nll_grad':
            xg = x.clone().requires_grad_(True)
            flow.zero_grad()
            loss = -flow.log_prob(xg, **kw).mean()
            loss.backward()
            out['nll.loss'] = loss.detach()
            out['nll.grad_x'] = xg.grad
            for i, p in enumerate(flow.parameters()):
                out[f'nll.grad_p{i}'] = p.grad
        else:
            raise ValueError(op)
    torch.set_default_dtype(torch.float32)
    return {k: v.detach().cpu().numpy() for k, v in out.items()}


def main():
    blob = {}
    only = [a for a in sys.argv[1:] if not a.startswith('-')]
    if only:
        # python make_golden.py CASE [CASE ...]: record just these cases and merge them into the existing file
        path = os.path.join(HERE, 'reference_outputs.npz')
        blob = dict(np.load(path))
        for name in only:
            r32 = run_case(name, torch.float32)
            r64 = run_case(name, torch.float64)
            for k, v in r32.items():
                blob[f'{name}|{k}|f32'] = v
            for k, v in r64.items():
                if not k.endswith('.bins'):
                    blob[f'{name}|{k}|f64'] = v
            print(name, sorted(r32))
        np.savez_compressed(path, **sample_large(blob))
        print('merged into', path, len(blob), 'arrays', os.path.getsize(path), 'bytes')
        return
    for name in cases.CASES:
        r32 = run_case(name, torch.float32)
        r64 = run_case(name, torch.float64)
        for k, v in r32.items():
            blob[f'{name}|{k}|f32'] = v
        for k, v in r64.items():
            if k.endswith('.bins'):
                continue
            blob[f'{name}|{k}|f64'] = v
        print(name, sorted(r32))

    # the reference's own golden vector (flow.py:77-84, test_normalizing_flow.py:45-55):
    # seeded with torch's RNG exactly as the reference test does.
    torch.manual_seed(123)
    f = st.NormalizingFlow(st.UnitNormal(2), [st.Affine(2)])
    aff = f.transforms[0]
    y = torch.randn(3, 2)
    blob['doc_example|log_scale|f32'] = aff.log_scale.detach().numpy().copy()
    blob['doc_example|shift|f32'] = aff.shift.detach().numpy().copy()
    blob['doc_example|y|f32'] = y.numpy().copy()
    blob['doc_example|log_prob|f32'] = f.log_prob(y).detach().numpy()
    z = torch.randn(1, 2)      # what base_dist.sample((1,)) would consume is torch-RNG specific;
    blob['doc_example|z|f32'] = z.numpy().copy()      # store an explicit latent draw instead
    blob['doc_example|forward_z|f32'] = f.forward(z).detach().numpy()

    # exact mask vectors (util/mask.py) for a range of dims
    for nm in ('none', 'ordered_right_half', 'ordered_0', 'ordered_left_half', 'ordered_1',
               'parity_even', 'parity_odd'):
        gen = st.util.get_mask(nm)
        for d in (1, 2, 3, 5, 16, 64, 127, 128):
            blob[f'mask|{nm}|{d}'] = gen(d).numpy()

    path = os.path.join(HERE, 'reference_outputs.npz')
    np.savez_compressed(path, **sample_large(blob))
    print('wrote', path, len(blob), 'arrays', os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
