"""ctypes binding of libstribor_b200.so (the C ABI declared in include/stribor_b200.h).

There is deliberately NO fallback: if the shared library is missing or a call fails the
caller gets an exception.  Build it with ``python -c "import __graft_entry__ as g; g.build()"``
(or ``python -m stribor_b200.build``).
"""
from __future__ import annotations

import ctypes as C
import os

STB_MAX_LINEAR = 8
ABI_VERSION = 3

# enums (include/stribor_b200.h)
AFFINE, RQS, CUBIC, CONT_AFFINE, PERMUTE, SIGMOID, LOGIT = 0, 1, 2, 3, 4, 5, 6
FORWARD, INVERSE = 0, 1
LDJ_NONE, LDJ_SET, LDJ_ADD = 0, 1, 2
ACTIVATIONS = {None: 0, 'Identity': 0, 'Tanh': 1, 'ReLU': 2, 'Sigmoid': 3, 'ELU': 4, 'Softplus': 5,
               'LeakyReLU': 6, 'SiLU': 7, 'GELU': 8}
E_INVAL, E_CUDA, E_NOTSUP = -1, -2, -3

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'libstribor_b200.so')

EXPORTS = ['stb_abi_version', 'stb_sizeof_layer', 'stb_last_error', 'stb_layer_apply', 'stb_layer_apply_diag',
           'stb_layer_apply_bins', 'stb_flow_apply',
           'stb_flow_log_prob', 'stb_flow_log_prob_needs_x_out', 'stb_unit_normal_log_prob', 'stb_layer_backward_workspace_bytes',
           'stb_layer_backward', 'stb_layer_backward_diag', 'stb_packed_bytes', 'stb_pack_layer', 'stb_layer_uses_tensor_path',
           'stb_launch_count', 'stb_tc_selftest']


class StbMlp(C.Structure):
    _fields_ = [('n_linear', C.c_int32), ('activation', C.c_int32), ('final_activation', C.c_int32),
                ('dims', C.c_int32 * (STB_MAX_LINEAR + 1)),
                ('W', C.c_void_p * STB_MAX_LINEAR), ('b', C.c_void_p * STB_MAX_LINEAR)]


class StbSplineOpts(C.Structure):
    _fields_ = [('custom', C.c_int32), ('min_bin_width', C.c_float), ('min_bin_height', C.c_float),
                ('min_derivative', C.c_float), ('free_edge_derivs', C.c_int32),
                ('cub_eps', C.c_float), ('cub_quad_threshold', C.c_float)]


class StbLayer(C.Structure):
    _fields_ = [('kind', C.c_int32), ('dim', C.c_int32), ('latent_dim', C.c_int32),
                ('cond_x', C.c_int32), ('time_input', C.c_int32), ('n_bins', C.c_int32),
                ('inverse_ldj_own', C.c_int32), ('zero_cond', C.c_int32),
                ('lower', C.c_float), ('upper', C.c_float),
                ('left', C.c_float), ('right', C.c_float), ('bottom', C.c_float), ('top', C.c_float),
                ('has_box', C.c_int32), ('row_compact', C.c_int32),
                ('mask', C.c_void_p), ('mask_host', C.c_void_p), ('const_out', C.c_void_p), ('row_out', C.c_void_p),
                ('time_scale', C.c_void_p), ('perm', C.c_void_p), ('perm_inv', C.c_void_p),
                ('net', StbMlp), ('packed', C.c_void_p), ('packed_bytes', C.c_uint64),
                ('perm_host', C.c_void_p), ('perm_inv_host', C.c_void_p), ('spline', StbSplineOpts)]


class StbLayerGrads(C.Structure):
    _fields_ = [('gW', C.c_void_p * STB_MAX_LINEAR), ('gb', C.c_void_p * STB_MAX_LINEAR),
                ('g_const_out', C.c_void_p), ('g_time_scale', C.c_void_p), ('g_row_out', C.c_void_p)]


class StriborB200Error(RuntimeError):
    pass


_lib = None


def lib():
    """Load the shared library once; raise loudly if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise StriborB200Error(
            f'{LIB_PATH} not found: the CUDA extension has not been built. '
            'There is no CPU / PyTorch fallback -- run `python -m stribor_b200.build`.')
    l = C.CDLL(LIB_PATH)
    vp, i32, i64, u64 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64
    LP = C.POINTER(StbLayer)
    l.stb_abi_version.restype = i32
    l.stb_last_error.restype = C.c_char_p
    l.stb_launch_count.restype = u64
    l.stb_layer_apply.restype = i32
    l.stb_layer_apply.argtypes = [LP, i32, vp, vp, vp, vp, vp, i32, i32, i64, vp]
    l.stb_layer_apply_bins.restype = i32
    l.stb_layer_apply_bins.argtypes = [LP, i32, vp, vp, vp, vp, vp, i32, vp, i64, vp]
    l.stb_layer_apply_diag.restype = i32
    l.stb_layer_apply_diag.argtypes = [LP, i32, vp, vp, vp, vp, vp, i64, vp]
    l.stb_flow_apply.restype = i32
    l.stb_flow_apply.argtypes = [LP, i32, i32, vp, vp, vp, vp, vp, i32, i64, vp]
    l.stb_flow_log_prob.restype = i32
    l.stb_flow_log_prob.argtypes = [LP, i32, vp, vp, vp, vp, vp, i64, vp]
    l.stb_flow_log_prob_needs_x_out.restype = i32
    l.stb_flow_log_prob_needs_x_out.argtypes = [LP, i32]
    l.stb_unit_normal_log_prob.restype = i32
    l.stb_unit_normal_log_prob.argtypes = [vp, vp, i32, C.c_int32, i64, vp]
    l.stb_layer_backward_workspace_bytes.restype = u64
    l.stb_layer_backward_workspace_bytes.argtypes = [LP, i64]
    l.stb_layer_backward.restype = i32
    l.stb_layer_backward.argtypes = [LP, i32, vp, vp, vp, vp, vp, vp, vp, vp,
                                     C.POINTER(StbLayerGrads), vp, i64, vp]
    l.stb_layer_backward_diag.restype = i32
    l.stb_layer_backward_diag.argtypes = [LP, i32, vp, vp, vp, vp, C.POINTER(StbLayerGrads), i64, vp]
    l.stb_packed_bytes.restype = u64
    l.stb_packed_bytes.argtypes = [LP]
    l.stb_pack_layer.restype = i32
    l.stb_pack_layer.argtypes = [LP, vp, vp]
    l.stb_layer_uses_tensor_path.restype = i32
    l.stb_layer_uses_tensor_path.argtypes = [LP]
    l.stb_tc_selftest.restype = i32
    l.stb_tc_selftest.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp]
    l.stb_sizeof_layer.restype = u64
    if l.stb_sizeof_layer() != C.sizeof(StbLayer):
        raise StriborB200Error(f'stb_layer layout mismatch: C {l.stb_sizeof_layer()} vs ctypes {C.sizeof(StbLayer)}')
    if l.stb_abi_version() != ABI_VERSION:
        raise StriborB200Error(f'ABI mismatch: library {l.stb_abi_version()} vs binding {ABI_VERSION}')
    _lib = l
    return l


def check(rc: int):
    """Map a negative return code to the exception type the reference raises for that class
    of problem (SURVEY.md section 8b): bad configuration -> ValueError, not built ->
    NotImplementedError, CUDA failure -> RuntimeError."""
    if rc == 0:
        return
    msg = lib().stb_last_error().decode('utf-8', 'replace')
    if rc == E_INVAL:
        raise ValueError(msg)
    if rc == E_NOTSUP:
        raise NotImplementedError(msg)
    raise StriborB200Error(f'stribor_b200 error {rc}: {msg}')
