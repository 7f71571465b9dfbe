"""torch.library custom ops in front of the C ABI.

Python owns the tensors (allocation, streams, autograd graph); the arithmetic happens in
libstribor_b200.so.  Three ops:

  stribor_b200::layer_apply     one layer, one direction (+ log|det J|), differentiable
  stribor_b200::layer_backward  its gradient (recompute-from-input)
  stribor_b200::flow_chain      a whole chain of layers in one C call (inference fast path:
                                forward / inverse / log_prob incl. the UnitNormal term)

A layer is described by plain data so that it can cross the op boundary:
  meta  = [kind, dim, latent_dim, cond_x, time_input, n_bins, inverse_ldj_own, zero_cond,
           activation, final_activation, n_linear, n_params, has_box, row_mode, dims[0..n_linear],
           mask[0..dim) (only when cond_x)]
  fmeta = [lower, upper, left, right, bottom, top] (+ [custom, min_bin_width, min_bin_height, min_derivative,
           free_edge_derivs, cub_eps, cub_quad_threshold]: stb_spline_opts, functional spline API only;
           without them the reference defaults)
  params = [W0, b0, W1, b1, ...] (+ [time_scale]) or [const_out]   (row_mode: const_out is a
           per-row [rows, out_width] tensor -> stb_layer.row_out; row_mode 2 = compact: only the
           transformed dims' parameters, [rows, n_tr * P])
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib

META_HEADER = 14
FMETA_LEN = 6
SPLINE_OPTS_LEN = 7


DTYPES = {torch.float32: _lib.F32, torch.float64: _lib.F64}


def _check_cuda(x: Tensor, what: str):
    if not x.is_cuda:
        raise RuntimeError(
            f'stribor_b200: {what} is on {x.device}; this package runs its transforms in CUDA '
            'kernels only (sm_100a) and has no CPU fallback -- move the module and inputs to a GPU.')
    if x.dtype not in DTYPES:
        raise TypeError(f'stribor_b200: {what} must be float32 or float64, got {x.dtype}')


def check_layer_tensors(x: Tensor, latent: Optional[Tensor], t: Optional[Tensor], mask: Optional[Tensor],
                        params: Sequence[Tensor], packed: Optional[Tensor] = None, int_params: bool = False):
    """Every tensor whose raw pointer is handed to the kernels must live on x's device with the dtype the
    kernels read -- x's, float32 or float64, for every floating tensor of the call (mixed dtypes are not
    promoted): a float64 ``t`` / ``latent`` next to a float32 input would be reinterpreted as float32 pairs, a
    module left on the CPU (or another GPU) would hand a foreign pointer to the kernel.  Raise the
    reference-style Python error instead."""
    _check_cuda(x, 'input')
    dev = x.device

    def same(v, what, dtype):
        if v is None or v.numel() == 0:
            return
        if v.device != dev:
            raise RuntimeError(f'stribor_b200: {what} is on {v.device} but the input is on {dev}; move the module '
                               'and all inputs to the same GPU (there is no CPU fallback)')
        if v.dtype != dtype:
            raise TypeError(f'stribor_b200: {what} must be {dtype}, got {v.dtype}')
        if not v.is_contiguous():
            raise ValueError(f'stribor_b200: {what} must be contiguous')

    same(latent, '`latent`', x.dtype)
    same(t, '`t`', x.dtype)
    same(mask, 'the coupling mask', torch.uint8)
    for i, p in enumerate(params):
        same(p, f'layer parameter {i}', torch.int32 if int_params else x.dtype)
    same(packed, 'the packed weight image', torch.uint8)


def _dp(t: Optional[Tensor]):
    return None if t is None or t.numel() == 0 else t.data_ptr()


def _stream(x: Tensor):
    return torch.cuda.current_stream(x.device).cuda_stream


def _fill_struct(L: _lib.StbLayer, meta: Sequence[int], fmeta: Sequence[float], mask: Optional[Tensor],
                 params: Sequence[Tensor], packed: Optional[Tensor], dtype: torch.dtype = torch.float32):
    """``dtype``: the input tensor's, which every float pointer of the call points to (stb_layer.dtype)."""
    (kind, dim, latent_dim, cond_x, time_input, n_bins, inv_own, zero_cond, act, fact, n_linear,
     n_params, has_box, row_mode) = meta[:META_HEADER]
    L.kind, L.dim, L.latent_dim, L.cond_x = kind, dim, latent_dim, cond_x
    L.time_input, L.n_bins, L.inverse_ldj_own, L.zero_cond = time_input, n_bins, inv_own, zero_cond
    L.lower, L.upper = float(fmeta[0]), float(fmeta[1])
    L.left, L.right, L.bottom, L.top = (float(v) for v in fmeta[2:6])
    L.has_box = has_box
    L.dtype = DTYPES[dtype]
    if len(fmeta) > FMETA_LEN:
        custom, mw, mh, md, free_edge, eps, quad = fmeta[FMETA_LEN:FMETA_LEN + SPLINE_OPTS_LEN]
        o = L.spline
        o.custom, o.free_edge_derivs = int(custom), int(free_edge)
        o.min_bin_width, o.min_bin_height, o.min_derivative = float(mw), float(mh), float(md)
        o.cub_eps, o.cub_quad_threshold = float(eps), float(quad)
    L.row_compact = 1 if row_mode == 2 else 0
    L.mask = _dp(mask)
    keep = None
    if cond_x:
        off = META_HEADER + (n_linear + 1 if n_linear > 0 else 0)
        keep = (C.c_uint8 * dim)(*meta[off:off + dim])
        L.mask_host = C.cast(keep, C.c_void_p)
    else:
        L.mask_host = None
    L.net.n_linear = n_linear
    L.net.activation = act
    L.net.final_activation = fact
    assert len(params) == n_params, (len(params), n_params)
    if n_linear > 0:
        dims = meta[META_HEADER:META_HEADER + n_linear + 1]
        for i, v in enumerate(dims):
            L.net.dims[i] = v
        for i in range(n_linear):
            w, b = params[2 * i], params[2 * i + 1]
            assert w.is_contiguous() and b.is_contiguous()
            assert tuple(w.shape) == (dims[i + 1], dims[i]), (tuple(w.shape), dims)
            L.net.W[i] = w.data_ptr()
            L.net.b[i] = b.data_ptr()
        rest = params[2 * n_linear:]
        L.const_out = None
        L.row_out = None
    elif kind >= _lib.PERMUTE:
        L.const_out = L.row_out = None
        rest = params
    else:
        assert params[0].is_contiguous()
        L.const_out = None if row_mode else params[0].data_ptr()
        L.row_out = params[0].data_ptr() if row_mode else None
        rest = params[1:]
    L.time_scale = rest[0].data_ptr() if kind == _lib.CONT_AFFINE else None
    L.perm_host = L.perm_inv_host = None
    if kind == _lib.PERMUTE:                      # params = [perm (int32), perm_inv (int32)]
        L.const_out = None
        L.perm, L.perm_inv = params[0].data_ptr(), params[1].data_ptr()
        if len(meta) >= META_HEADER + 2 * dim:    # host copies ride in the meta list: [perm(dim) | perm_inv(dim)]
            hp = (C.c_int32 * dim)(*meta[META_HEADER:META_HEADER + dim])
            hi = (C.c_int32 * dim)(*meta[META_HEADER + dim:META_HEADER + 2 * dim])
            L.perm_host, L.perm_inv_host = C.cast(hp, C.c_void_p), C.cast(hi, C.c_void_p)
            keep = (hp, hi)
    else:
        L.perm = L.perm_inv = None
    if packed is not None and packed.numel() > 0:
        L.packed = packed.data_ptr()
        L.packed_bytes = packed.numel() * packed.element_size()
    else:
        L.packed = None
        L.packed_bytes = 0
    return keep


def make_struct(meta, fmeta, mask, params, packed=None, dtype=torch.float32) -> _lib.StbLayer:
    L = _lib.StbLayer()
    L._keepalive = _fill_struct(L, meta, fmeta, mask, params, packed, dtype)
    return L


def meta_len(meta: Sequence[int], off: int = 0) -> int:
    n_linear = meta[off + 10]
    return META_HEADER + (n_linear + 1 if n_linear > 0 else 0) + (meta[off + 1] if meta[off + 3] else 0) + \
        (2 * meta[off + 1] if meta[off] == _lib.PERMUTE else 0)


# ----------------------------------------------------------------------------------------------
# one layer
# ----------------------------------------------------------------------------------------------
@torch.library.custom_op('stribor_b200::layer_apply', mutates_args=(), device_types='cuda')
def layer_apply(x: Tensor, latent: Optional[Tensor], t: Optional[Tensor], mask: Optional[Tensor],
                params: List[Tensor], packed: Optional[Tensor], meta: List[int], fmeta: List[float],
                direction: int, want_ldj: bool, base_lp: bool) -> Tuple[Tensor, Tensor]:
    """x [rows, dim] -> (y [rows, dim], ldj [rows] or empty)."""
    rows, dim = x.shape
    y = torch.empty_like(x)
    ldj = torch.empty(rows if want_ldj else 0, dtype=x.dtype, device=x.device)
    if rows == 0:
        return y, ldj
    L = make_struct(meta, fmeta, mask, params, packed, x.dtype)
    with torch.cuda.device(x.device):
        rc = _lib.lib().stb_layer_apply(C.byref(L), direction, x.data_ptr(), _dp(latent), _dp(t),
                                        y.data_ptr(), _dp(ldj), _lib.LDJ_SET if want_ldj else _lib.LDJ_NONE,
                                        int(base_lp), rows, _stream(x))
    _lib.check(rc)
    return y, ldj


@layer_apply.register_fake
def _(x, latent, t, mask, params, packed, meta, fmeta, direction, want_ldj, base_lp):
    return torch.empty_like(x), x.new_empty(x.shape[0] if want_ldj else 0)


@torch.library.custom_op('stribor_b200::layer_apply_diag', mutates_args=(), device_types='cuda')
def layer_apply_diag(x: Tensor, latent: Optional[Tensor], t: Optional[Tensor], mask: Optional[Tensor],
                     params: List[Tensor], meta: List[int], fmeta: List[float], direction: int
                     ) -> Tuple[Tensor, Tensor]:
    """x [rows, dim] -> (y [rows, dim], per-dimension log-derivative [rows, dim]).  Differentiable when the
    layer's parameters are supplied (const_out / row_out), see ``layer_backward_diag``."""
    rows, dim = x.shape
    y = torch.empty_like(x)
    ldiag = torch.empty_like(x)
    if rows == 0:
        return y, ldiag
    L = make_struct(meta, fmeta, mask, params, None, x.dtype)
    with torch.cuda.device(x.device):
        rc = _lib.lib().stb_layer_apply_diag(C.byref(L), direction, x.data_ptr(), _dp(latent), _dp(t),
                                             y.data_ptr(), ldiag.data_ptr(), rows, _stream(x))
    _lib.check(rc)
    return y, ldiag


@layer_apply_diag.register_fake
def _(x, latent, t, mask, params, meta, fmeta, direction):
    return torch.empty_like(x), torch.empty_like(x)



def _const_param_slabs(rows: int, numel: int):
    """Row ranges for the gradient of a broadcast (learned, ``[1, dim * P]``) parameter: the kernels write one
    gradient row per input row, which is then summed -- in slabs of at most 256 MB instead of a dense
    ``[rows, dim * P]`` tensor (12 GB at 1 M rows, dim 64, 47 parameters)."""
    slab = max(4096, (256 << 20) // (4 * max(numel, 1)))
    return [(s0, min(slab, rows - s0)) for s0 in range(0, rows, slab)]


def _off(ptr, count, width=1, esize=4):
    return None if ptr is None else ptr + esize * count * width


@torch.library.custom_op('stribor_b200::layer_backward_diag', mutates_args=(), device_types='cuda')
def layer_backward_diag(x: Tensor, mask: Optional[Tensor], params: List[Tensor], meta: List[int],
                        fmeta: List[float], direction: int, g_y: Tensor, g_ld: Optional[Tensor]) -> List[Tensor]:
    """Gradient of ``layer_apply_diag`` (``stb_layer_backward_diag``) -> [g_x, g_param]."""
    rows, dim = x.shape
    n_linear, row_mode = meta[10], meta[13]
    if n_linear > 0:
        raise NotImplementedError('stribor_b200: the per-dimension log-derivative API is differentiable when the '
                                  'transform parameters are tensors (learned, or a conditioner evaluated by autograd)')
    p0 = params[0]
    g_x = torch.empty_like(x)
    if rows == 0:
        return [g_x, torch.zeros_like(p0)]
    L = make_struct(meta, fmeta, mask, params, None, x.dtype)
    G = _lib.StbLayerGrads()
    lib = _lib.lib()
    if row_mode:
        g_rows = torch.zeros_like(p0)
        G.g_row_out = g_rows.data_ptr()
        with torch.cuda.device(x.device):
            _lib.check(lib.stb_layer_backward_diag(C.byref(L), direction, x.data_ptr(), g_y.data_ptr(), _dp(g_ld),
                                                   g_x.data_ptr(), C.byref(G), rows, _stream(x)))
        return [g_x, g_rows]
    slabs = _const_param_slabs(rows, p0.numel())
    g_rows = x.new_empty(slabs[0][1], p0.numel())
    g_p = x.new_zeros(p0.numel())
    G.g_row_out = g_rows.data_ptr()
    es = x.element_size()
    with torch.cuda.device(x.device):
        for s0, n in slabs:
            g_rows[:n].zero_()
            _lib.check(lib.stb_layer_backward_diag(C.byref(L), direction, _off(x.data_ptr(), s0, dim, es), _off(g_y.data_ptr(), s0, dim, es),
                                                   _off(_dp(g_ld), s0, dim, es), _off(g_x.data_ptr(), s0, dim, es), C.byref(G), n, _stream(x)))
            g_p += g_rows[:n].sum(0)
    return [g_x, g_p.view_as(p0)]


@layer_backward_diag.register_fake
def _(x, mask, params, meta, fmeta, direction, g_y, g_ld):
    return [torch.empty_like(x), torch.empty_like(params[0])]


def _setup_ctx_diag(ctx, inputs, output):
    x, latent, t, mask, params, meta, fmeta, direction = inputs
    ctx.save_for_backward(x, mask, *params)
    ctx.meta, ctx.fmeta, ctx.direction = list(meta), list(fmeta), direction


def _backward_diag(ctx, g_y, g_ld):
    saved = ctx.saved_tensors
    x, mask = saved[:2]
    params = list(saved[2:])
    g_y = g_y.contiguous() if g_y is not None else torch.zeros_like(x)
    g_ld = g_ld.contiguous() if g_ld is not None else None
    g_x, g_p = layer_backward_diag(x, mask, params, ctx.meta, ctx.fmeta, ctx.direction, g_y, g_ld)
    return g_x, None, None, None, [g_p] + [None] * (len(params) - 1), None, None, None


layer_apply_diag.register_autograd(_backward_diag, setup_context=_setup_ctx_diag)


def layer_apply_bins(x: Tensor, latent: Optional[Tensor], t: Optional[Tensor], mask: Optional[Tensor],
                     params: List[Tensor], packed: Optional[Tensor], meta: List[int], fmeta: List[float],
                     direction: int) -> Tuple[Tensor, Tensor, Tensor]:
    """Parity instrument (``stb_layer_apply_bins``): x [rows, dim] -> (y, ldj [rows], bins [rows, dim] int32).
    ``bins`` is the bin each element's knot search chose on the SAME kernel path ``layer_apply`` takes
    (tensor-core kernels when ``packed`` is given); -1 for pass-through dims and identity tails."""
    _check_cuda(x, 'input')
    rows, dim = x.shape
    y = torch.empty_like(x)
    ldj = torch.empty(rows, dtype=x.dtype, device=x.device)
    bins = torch.full((rows, dim), -1, dtype=torch.int32, device=x.device)
    if rows == 0:
        return y, ldj, bins
    L = make_struct(meta, fmeta, mask, params, packed, x.dtype)
    with torch.cuda.device(x.device):
        rc = _lib.lib().stb_layer_apply_bins(C.byref(L), direction, x.data_ptr(), _dp(latent), _dp(t),
                                             y.data_ptr(), ldj.data_ptr(), _lib.LDJ_SET, bins.data_ptr(),
                                             rows, _stream(x))
    _lib.check(rc)
    return y, ldj, bins


G_PAD = 48            # parameters per transformed dim in g_net (47 quadratic, padded)
H_AUG = 72            # workspace row: hidden(64) | 1 | 0 x 7


_PACKED_COLS = {}


def _packed_cols(dev):
    """Natural parameter index [w(16) | h(16) | d(15) | pad] -> column of the kernels' packed order
    ((w_i, h_i) interleaved, then the derivative columns)."""
    k = str(dev)
    if k not in _PACKED_COLS:
        cols = [2 * p for p in range(16)] + [2 * p + 1 for p in range(16)] + list(range(32, 48))
        _PACKED_COLS[k] = torch.tensor(cols, dtype=torch.long, device=dev)
    return _PACKED_COLS[k]


_INDEX_CACHE = {}


def _index_tensors(mask_tuple, dev):
    """(transformed columns, conditioning columns) of a mask as device index tensors, cached: building them
    per call is a blocking host-to-device copy in the middle of the backward pass."""
    k = (mask_tuple, str(dev))
    if k not in _INDEX_CACHE:
        tr = [j for j, m in enumerate(mask_tuple) if m == 0]
        cond = [j for j, m in enumerate(mask_tuple) if m != 0]
        _INDEX_CACHE[k] = (torch.tensor(tr, dtype=torch.long, device=dev), torch.tensor(cond, dtype=torch.long, device=dev))
    return _INDEX_CACHE[k]


def fused_backward_ok(L: '_lib.StbLayer') -> bool:
    """Does stb_layer_backward differentiate this (packed) layer with its conditioner fused?"""
    return int(_lib.lib().stb_layer_backward_workspace_bytes(C.byref(L), 1)) > 0


def _fused_conditioner_backward(x, mask, params, packed, meta, fmeta, direction, g_y, g_ldj):
    """Coupling(Spline, MLP[64]) on the tensor-core path: ONE kernel (stb_layer_backward -> tc_wide.cu) recomputes
    the conditioner from the saved input, differentiates the spline in registers and forms the conditioner's
    gradient products on the tensor cores.  Three arrangements, selected by environment (default first):
      fused           g_x complete; images of [gW2 | gb2], gW1 (conditioning slots) and gb1 come back in the
                      workspace -- nothing left here but un-packing them
      ..W1_LIB=1      as above without the first Linear: g_pre [rows, 64] comes back and
                      gW1 = g_pre^T x_cond, gb1 = sum g_pre, g_x[cond] += g_pre W1[:, cond] are library GEMMs
      ..GNET=1        two-step (quadratic only): g_net [rows, n_tr * 48] and [hidden | 1] come back, all four
                      products are fp32 library GEMMs"""
    rows, dim = x.shape
    W1, b1, W2, b2 = params
    act = meta[8]
    off = META_HEADER + meta[10] + 1
    mask_list = meta[off:off + dim]
    tr = [j for j, m in enumerate(mask_list) if m == 0]
    cond = [j for j, m in enumerate(mask_list) if m != 0]
    n_tr, P = len(tr), W2.shape[0] // dim
    g_x = torch.empty_like(x)
    gW1, gb1, gW2, gb2 = torch.zeros_like(W1), torch.zeros_like(b1), torch.zeros_like(W2), torch.zeros_like(b2)
    if rows == 0:
        g_x.zero_()
        return [g_x, x.new_empty(0), x.new_empty(0), gW1, gb1, gW2, gb2]
    L = make_struct(meta, fmeta, mask, params, packed, x.dtype)
    lib = _lib.lib()
    ws_bytes = int(lib.stb_layer_backward_workspace_bytes(C.byref(L), rows)) if packed is not None else 0
    if act not in (_lib.ACTIVATIONS['Tanh'], _lib.ACTIVATIONS['Sigmoid'], _lib.ACTIVATIONS['ReLU']):
        ws_bytes = 0
    if ws_bytes == 0:
        raise NotImplementedError('stribor_b200: this layer has no fused conditioner backward '
                                  '(quadratic spline, 16 bins, MLP[64], dim <= 128 on the tensor-core path)')
    dev = x.device
    tr_t, cond_t = _index_tensors(tuple(mask_list), dev)
    hid = W2.shape[1]
    G = _lib.StbLayerGrads()
    if os.environ.get('STRIBOR_B200_TRAIN_GNET') == '1' and meta[0] == _lib.RQS:
        # two-step variant: the kernel leaves g_net / [hidden | 1]; the last Linear's products are library GEMMs
        g_net = torch.empty(rows, n_tr * G_PAD, dtype=x.dtype, device=dev)
        ws = torch.empty(ws_bytes // 4, dtype=x.dtype, device=dev)
        haug = ws[:rows * H_AUG].view(rows, H_AUG)
        G.g_row_out = g_net.data_ptr()
        with torch.cuda.device(dev):
            rc = lib.stb_layer_backward(C.byref(L), direction, x.data_ptr(), None, None, g_y.data_ptr(), _dp(g_ldj),
                                        g_x.data_ptr(), None, None, C.byref(G), ws.data_ptr(), rows, _stream(x))
        _lib.check(rc)
        W2p = W2.new_zeros(n_tr, G_PAD, hid)
        W2p[:, :P] = W2.view(dim, P, hid).index_select(0, tr_t)
        gaug = (g_net.t() @ haug).view(n_tr, G_PAD, H_AUG)      # [gW2 | gb2 | 0] of the transformed dims' rows
        gW2.view(dim, P, hid).index_copy_(0, tr_t, gaug[:, :P, :hid].contiguous())
        gb2.view(dim, P).index_copy_(0, tr_t, gaug[:, :P, hid].contiguous())
        h = haug[:, :hid]
        g_h = g_net @ W2p.view(n_tr * G_PAD, hid)
        if act == _lib.ACTIVATIONS['Tanh']:
            g_pre = g_h * (1.0 - h * h)
        elif act == _lib.ACTIVATIONS['Sigmoid']:
            g_pre = g_h * (h * (1.0 - h))
        else:
            g_pre = g_h * (h > 0).to(g_h.dtype)
    else:
        # fused: the [gW2 | gb2] image (packed column order) comes out of the kernel; by default also the first
        # Linear's gradients and the complete g_x (STRIBOR_B200_TRAIN_W1_LIB=1: those three K = 64 products as
        # library GEMMs from g_pre, the previous arrangement)
        w1_in_kernel = os.environ.get('STRIBOR_B200_TRAIN_W1_LIB') != '1'
        ws = torch.empty(ws_bytes // 4, dtype=x.dtype, device=dev)
        img = ws[rows * H_AUG:]
        img.zero_()
        with torch.cuda.device(dev):
            rc = lib.stb_layer_backward(C.byref(L), direction, x.data_ptr(), None, None, g_y.data_ptr(), _dp(g_ldj),
                                        g_x.data_ptr(), None, None, None if w1_in_kernel else C.byref(G),
                                        ws.data_ptr(), rows, _stream(x))
        _lib.check(rc)
        n_pad = 2 * ((n_tr + 1) // 2)
        n_img = 64 * G_PAD * H_AUG
        nat = img[:n_img].view(-1, G_PAD, H_AUG)[:n_pad].index_select(1, _packed_cols(dev))[:n_tr]   # natural parameter order
        gW2.view(dim, P, hid).index_copy_(0, tr_t, nat[:, :P, :hid].contiguous())
        gb2.view(dim, P).index_copy_(0, tr_t, nat[:, :P, hid].contiguous())
        if w1_in_kernel:
            w1c = img[n_img:n_img + hid * 64].view(hid, 64)
            if cond:
                gW1.index_copy_(1, cond_t, w1c[:, :len(cond)])
            gb1 = img[n_img + hid * 64:n_img + hid * 64 + hid].clone()
            return [g_x, x.new_empty(0), x.new_empty(0), gW1, gb1, gW2, gb2]
        g_pre = ws[:rows * hid].view(rows, hid)
    if cond:
        contiguous = cond[-1] - cond[0] + 1 == len(cond)            # ordered masks: a column range, no gathers
        if contiguous:
            c0, c1 = cond[0], cond[-1] + 1
            xc, W1c = x[:, c0:c1], W1[:, c0:c1]
        else:
            xc, W1c = x.index_select(1, cond_t), W1.index_select(1, cond_t)
        # g_pre^T x_cond is a [64, n_cond] product over `rows`: split the long reduction into slabs so the
        # library GEMM fills the GPU (one [64 x 64] output tile would run on a handful of SMs)
        slab = 4096
        if rows >= 4 * slab and rows % slab == 0 and contiguous:
            gw = torch.bmm(g_pre.view(rows // slab, slab, hid).transpose(1, 2),
                           x.view(rows // slab, slab, dim)[:, :, c0:c1]).sum(0)
        else:
            gw = g_pre.t() @ xc
        if contiguous:
            gW1[:, c0:c1] = gw
            g_x[:, c0:c1].addmm_(g_pre, W1c)
        else:
            gW1.index_copy_(1, cond_t, gw)
            g_x.index_add_(1, cond_t, g_pre @ W1c)
    gb1 = g_pre.sum(0)
    return [g_x, x.new_empty(0), x.new_empty(0), gW1, gb1, gW2, gb2]


@torch.library.custom_op('stribor_b200::layer_backward', mutates_args=(), device_types='cuda')
def layer_backward(x: Tensor, latent: Optional[Tensor], t: Optional[Tensor], mask: Optional[Tensor],
                   params: List[Tensor], packed: Optional[Tensor], meta: List[int], fmeta: List[float],
                   direction: int, g_y: Tensor, g_ldj: Optional[Tensor], need_latent: bool, need_t: bool
                   ) -> List[Tensor]:
    """-> [g_x, g_latent (or empty), g_t (or empty), *g_params]."""
    rows, dim = x.shape
    n_linear, row_mode = meta[10], meta[13]
    if n_linear > 0 and meta[0] != _lib.CONT_AFFINE:
        return _fused_conditioner_backward(x, mask, params, packed, meta, fmeta, direction, g_y, g_ldj)
    if n_linear > 0 or meta[0] == _lib.CONT_AFFINE:
        raise NotImplementedError(
            'stribor_b200: the continuous-affine conditioner backward is not built yet '
            '(training runs the MLP through autograd around the element-wise kernels)')
    g_x = torch.empty_like(x)
    g_latent = x.new_empty(0)
    g_t = x.new_empty(0)
    p0 = params[0]
    if rows == 0:
        g_x.zero_()
        return [g_x, g_latent, g_t, torch.zeros_like(p0)]
    # per-row gradient wrt the network output; a broadcast (const) parameter sums it over rows, slab by slab
    L = make_struct(meta, fmeta, mask, params, None, x.dtype)
    G = _lib.StbLayerGrads()
    lib = _lib.lib()
    if row_mode:
        g_rows = torch.zeros_like(p0)
        G.g_row_out = g_rows.data_ptr()
        with torch.cuda.device(x.device):
            _lib.check(lib.stb_layer_backward(C.byref(L), direction, x.data_ptr(), _dp(latent), _dp(t),
                                              g_y.data_ptr(), _dp(g_ldj), g_x.data_ptr(), None, None,
                                              C.byref(G), None, rows, _stream(x)))
        return [g_x, g_latent, g_t, g_rows]
    slabs = _const_param_slabs(rows, p0.numel())
    g_rows = x.new_empty(slabs[0][1], p0.numel())
    g_p = x.new_zeros(p0.numel())
    G.g_row_out = g_rows.data_ptr()
    lat_w = 0 if latent is None else latent.shape[-1]
    es = x.element_size()
    with torch.cuda.device(x.device):
        for s0, n in slabs:
            g_rows[:n].zero_()
            _lib.check(lib.stb_layer_backward(C.byref(L), direction, _off(x.data_ptr(), s0, dim, es), _off(_dp(latent), s0, lat_w, es),
                                              _off(_dp(t), s0, 1, es), _off(g_y.data_ptr(), s0, dim, es), _off(_dp(g_ldj), s0, 1, es),
                                              _off(g_x.data_ptr(), s0, dim, es), None, None, C.byref(G), None, n, _stream(x)))
            g_p += g_rows[:n].sum(0)
    return [g_x, g_latent, g_t, g_p.view_as(p0)]


@layer_backward.register_fake
def _(x, latent, t, mask, params, packed, meta, fmeta, direction, g_y, g_ldj, need_latent, need_t):
    gl = torch.empty_like(latent) if (need_latent and latent is not None) else x.new_empty(0)
    gt = torch.empty_like(t) if (need_t and t is not None) else x.new_empty(0)
    return [torch.empty_like(x), gl, gt] + [torch.empty_like(p) for p in params]


def _setup_ctx(ctx, inputs, output):
    x, latent, t, mask, params, packed, meta, fmeta, direction, want_ldj, base_lp = inputs
    if base_lp:
        raise RuntimeError('base_lp is an inference-only fusion')
    ctx.save_for_backward(x, latent, t, mask, packed, *params)
    ctx.n_params = len(params)
    ctx.meta, ctx.fmeta, ctx.direction, ctx.want_ldj = list(meta), list(fmeta), direction, want_ldj
    ctx.has_latent, ctx.has_t = latent is not None, t is not None


def _backward(ctx, g_y, g_ldj):
    saved = ctx.saved_tensors
    x, latent, t, mask, packed = saved[:5]
    params = list(saved[5:])
    need = ctx.needs_input_grad
    g_y = g_y.contiguous() if g_y is not None else torch.zeros_like(x)
    gl = g_ldj.contiguous() if (ctx.want_ldj and g_ldj is not None) else None
    outs = layer_backward(x, latent, t, mask, params, packed, ctx.meta, ctx.fmeta, ctx.direction, g_y, gl,
                          bool(ctx.has_latent and need[1]), bool(ctx.has_t and need[2]))
    g_x, g_latent, g_t = outs[:3]
    g_params = list(outs[3:])
    return (g_x, g_latent if (ctx.has_latent and need[1]) else None,
            g_t if (ctx.has_t and need[2]) else None, None, g_params, None, None, None, None, None, None)


layer_apply.register_autograd(_backward, setup_context=_setup_ctx)


# ----------------------------------------------------------------------------------------------
# whole chain in one C call (no autograd)
# ----------------------------------------------------------------------------------------------
CHAIN_FORWARD, CHAIN_INVERSE, CHAIN_LOG_PROB, CHAIN_LOG_PROB_ONLY = 0, 1, 2, 3


def build_layer_array(masks: List[Tensor], params: List[Tensor], packed: List[Tensor], meta: List[int],
                      fmeta: List[float], dtype: torch.dtype = torch.float32):
    """-> (ctypes array of stb_layer, objects that must outlive it); ``dtype`` is the input's."""
    n_layers = len(masks)
    arr = (_lib.StbLayer * n_layers)()
    keep = []
    mo = po = 0
    for i in range(n_layers):
        ml = meta_len(meta, mo)
        m = meta[mo:mo + ml]
        npar = m[11]
        keep.append(_fill_struct(arr[i], m, fmeta[FMETA_LEN * i:FMETA_LEN * (i + 1)], masks[i],
                                 params[po:po + npar], packed[i], dtype))
        mo += ml
        po += npar
    return arr, keep


def flow_chain_launch(arr, n_layers: int, x: Tensor, latent: Optional[Tensor], t: Optional[Tensor], mode: int,
                      want_ldj: bool) -> Tuple[Tensor, Tensor]:
    """One C call over a prepared layer array (see ``flow_chain_direct`` for the modes)."""
    rows, dim = x.shape
    need_vec = want_ldj or mode in (CHAIN_LOG_PROB, CHAIN_LOG_PROB_ONLY)
    ldj = torch.empty(rows if need_vec else 0, dtype=x.dtype, device=x.device)
    if rows == 0:
        return torch.empty_like(x), ldj
    lib = _lib.lib()
    # log_prob without the latent rows: when the whole flow is one chained launch nothing has to be written back
    # but the log-probabilities (mode LOG_PROB_ONLY returns an empty first tensor)
    skip_x = mode == CHAIN_LOG_PROB_ONLY and lib.stb_flow_log_prob_needs_x_out(arr, n_layers) == 0
    out = x.new_empty(0, dim) if skip_x else torch.empty_like(x)
    with torch.cuda.device(x.device):
        if mode in (CHAIN_LOG_PROB, CHAIN_LOG_PROB_ONLY):
            rc = lib.stb_flow_log_prob(arr, n_layers, x.data_ptr(), _dp(latent), _dp(t), _dp(out),
                                       ldj.data_ptr(), rows, _stream(x))
        else:
            rc = lib.stb_flow_apply(arr, n_layers, _lib.FORWARD if mode == CHAIN_FORWARD else _lib.INVERSE,
                                    x.data_ptr(), _dp(latent), _dp(t), out.data_ptr(), _dp(ldj),
                                    _lib.LDJ_SET if want_ldj else _lib.LDJ_NONE, rows, _stream(x))
    _lib.check(rc)
    if mode == CHAIN_LOG_PROB_ONLY and not skip_x:
        out = x.new_empty(0, dim)                  # the scratch was needed (several launches) but is not returned
    return out, ldj


def flow_chain_direct(x: Tensor, latent: Optional[Tensor], t: Optional[Tensor], masks: List[Tensor],
                      params: List[Tensor], packed: List[Tensor], meta: List[int], fmeta: List[float],
                      mode: int, want_ldj: bool) -> Tuple[Tensor, Tensor]:
    """mode FORWARD/INVERSE: (out [rows,dim], ldj [rows] or empty);
    mode LOG_PROB: (latent x [rows,dim], log_prob [rows])."""
    arr, keep = build_layer_array(masks, params, packed, meta, fmeta, x.dtype)
    out = flow_chain_launch(arr, len(masks), x, latent, t, mode, want_ldj)
    del keep
    return out


# The registered op is what torch.compile / the dispatcher see; eager callers (flow.run_chain) keep the prepared layer
# array and call flow_chain_launch: the chain path never needs autograd, and the dispatcher round trip plus the
# per-call description of every layer cost more host time than a small batch spends on the GPU (tools/host_overhead.py).
flow_chain = torch.library.custom_op('stribor_b200::flow_chain', mutates_args=(), device_types='cuda')(flow_chain_direct)


@flow_chain.register_fake
def _(x, latent, t, masks, params, packed, meta, fmeta, mode, want_ldj):
    need_vec = want_ldj or mode in (CHAIN_LOG_PROB, CHAIN_LOG_PROB_ONLY)
    return (x.new_empty(0, x.shape[1]) if mode == CHAIN_LOG_PROB_ONLY else torch.empty_like(x)), \
        x.new_empty(x.shape[0] if need_vec else 0)


def launch_count() -> int:
    return int(_lib.lib().stb_launch_count())
