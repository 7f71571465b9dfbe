"""CPU: host side of the float64 layers -- the C ABI's dtype field and what it admits.  No kernel is launched and no
device pointer is dereferenced: these entry points decide from the layer description alone."""
import ctypes as C

import pytest
import torch

from stribor_b200 import _lib, _ops


def _struct(dim, kind='quadratic', hidden=(64,), n_bins=16, dtype=torch.float64, act='Tanh'):
    """stb_layer of Coupling(Spline / Affine, MLP(dim, hidden, dim * P)) with an ordered mask; CPU weight tensors"""
    kinds = {'quadratic': _lib.RQS, 'cubic': _lib.CUBIC, 'affine': _lib.AFFINE}
    P = {'quadratic': 3 * n_bins - 1, 'cubic': 2 * n_bins + 2}.get(kind, 2)
    dims = [dim] + list(hidden) + [dim * P]
    mask_list = [0] * (dim // 2) + [1] * (dim - dim // 2)
    params = []
    for i in range(len(dims) - 1):
        params += [torch.zeros(dims[i + 1], dims[i], dtype=dtype), torch.zeros(dims[i + 1], dtype=dtype)]
    meta = [kinds[kind], dim, 0, 1, 0, n_bins, 0, 0, _lib.ACTIVATIONS[act], 0, len(dims) - 1, len(params), 0, 0] + \
        dims + mask_list
    mask = torch.tensor(mask_list, dtype=torch.uint8)
    L = _ops.make_struct(meta, [-4., 4., 0., 1., 0., 1.], mask, params, None, dtype)
    L._keep = (params, mask)
    return L


def test_abi_version_and_layout():
    lib = _lib.lib()
    assert lib.stb_abi_version() == _lib.ABI_VERSION == 4
    assert lib.stb_sizeof_layer() == C.sizeof(_lib.StbLayer)
    assert [f[0] for f in _lib.StbLayer._fields_][-2:] == ['spline', 'dtype']
    assert (_lib.F32, _lib.F64) == (0, 1)
    assert _lib.StbLayer().dtype == _lib.F32                 # zero-filled: fp32, as before the field existed
    assert _struct(8).dtype == _lib.F64 and _struct(8, dtype=torch.float32).dtype == _lib.F32


@pytest.mark.parametrize('kind', ['quadratic', 'cubic', 'affine'])
def test_float64_layers_take_no_tensor_core_path(kind):
    lib = _lib.lib()
    L32, L64 = _struct(64, kind, dtype=torch.float32), _struct(64, kind)
    assert lib.stb_packed_bytes(C.byref(L32)) > 0             # the fp32 twin has an image
    assert lib.stb_packed_bytes(C.byref(L64)) == 0
    L64.packed, L64.packed_bytes = 1 << 20, 1 << 30          # even a (bogus) image does not select one
    assert lib.stb_layer_uses_tensor_path(C.byref(L64)) == 0
    assert lib.stb_pack_layer(C.byref(L64), C.c_void_p(1 << 20), None) == _lib.E_INVAL
    assert 'fp64' in lib.stb_last_error().decode()
    assert lib.stb_layer_backward_workspace_bytes(C.byref(L64), 1000) == 0
    arr = (_lib.StbLayer * 2)(L64, L64)
    assert lib.stb_flow_log_prob_needs_x_out(arr, 2) == 1
    # n_linear > 0 backward: fused conditioner backward only, which is fp32 -- refused before any pointer is read
    rc = lib.stb_layer_backward(C.byref(L64), _lib.FORWARD, 1 << 20, None, None, 1 << 20, None, 1 << 20, None, None,
                                None, 1 << 20, 8, None)
    assert rc == _lib.E_NOTSUP


def test_unknown_dtype_and_mixed_chains_are_rejected():
    lib = _lib.lib()
    bad = _struct(8)
    bad.dtype = 2
    assert lib.stb_packed_bytes(C.byref(bad)) == 0
    rc = lib.stb_layer_apply(C.byref(bad), _lib.FORWARD, 1 << 20, None, None, 1 << 20, None, 0, 0, 8, None)
    assert rc == _lib.E_INVAL and 'dtype' in lib.stb_last_error().decode()
    arr = (_lib.StbLayer * 2)(_struct(8), _struct(8, dtype=torch.float32))
    for direction in (_lib.FORWARD, _lib.INVERSE):
        rc = lib.stb_flow_apply(arr, 2, direction, 1 << 20, None, None, 1 << 20, None, 0, 8, None)
        assert rc == _lib.E_INVAL and 'dtype' in lib.stb_last_error().decode()
    rc = lib.stb_flow_log_prob(arr, 2, 1 << 20, None, None, 1 << 20, 1 << 21, 8, None)
    assert rc == _lib.E_INVAL and 'dtype' in lib.stb_last_error().decode()


def test_float64_shared_memory_limit():
    """The CUDA-core tile holds its activations in shared memory: in fp64 the widest conditioner is half the fp32 one.
    A float64 MLP[512] does not fit (the error is raised before anything is launched)."""
    lib = _lib.lib()
    L = _struct(64, hidden=(512,))
    rc = lib.stb_layer_apply(C.byref(L), _lib.FORWARD, 1 << 20, None, None, 1 << 20, None, 0, 0, 8, None)
    with pytest.raises(NotImplementedError, match='shared memory'):
        _lib.check(rc)
    # d = 64, K = 16, MLP[256, 256]: 8 * (64 * 33 + 2 * 256 * 32 + 47 * 129 + 4 * 32 + 32) + 4 * 64 bytes
    need = 8 * (64 * 33 + 2 * 256 * 32 + 47 * 129 + 4 * 32 + 32) + 4 * 64
    assert need <= 227 * 1024 < 8 * (64 * 33 + 2 * 512 * 32 + 47 * 129 + 4 * 32 + 32) + 4 * 64

