"""Functional spline API (reference: stribor/util/rational_quadratic_spline.py:7-125,
stribor/util/cubic_spline.py:10-69): per-element parameters supplied by the caller, evaluated
by the same CUDA kernels as the modules (``stb_layer.row_out`` mode)."""
from __future__ import annotations

import torch

from .. import _lib, _ops

__all__ = ['quadratic_spline_latent_dim', 'cubic_spline_latent_dim',
           'unconstrained_rational_quadratic_spline', 'unconstrained_cubic_spline']


def quadratic_spline_latent_dim(dim: int, n_bins: int) -> int:
    return dim * (3 * n_bins - 1)


def cubic_spline_latent_dim(dim: int, n_bins: int) -> int:
    return dim * (2 * n_bins + 2)


RQS_DEFAULTS = (1e-3, 1e-3, 1e-3)             # min_bin_width, min_bin_height, min_derivative
CUBIC_DEFAULTS = (1e-2, 1e-2, 1e-5, 1e-3)      # min_bin_width, min_bin_height, eps, quadratic_threshold


def _row_params_call(kind, inputs, pieces, n_bins, inverse, fmeta, has_box):
    _ops._check_cuda(inputs, 'inputs')
    shape = inputs.shape
    dim = shape[-1]
    x = inputs.reshape(-1, dim).contiguous()
    for p in pieces:
        if p.dtype != inputs.dtype:
            raise TypeError(f'stribor_b200: spline parameters must be {inputs.dtype} like the inputs, got {p.dtype}')
    prm = torch.cat([p.expand(*shape, p.shape[-1]) for p in pieces], -1).reshape(x.shape[0], -1).contiguous()
    meta = [kind, dim, 0, 0, 0, n_bins, 1, 0, 0, 0, 0, 1, int(has_box), 1]
    y, ld = _ops.layer_apply_diag(x, None, None, None, [prm], meta, fmeta,
                                  _lib.INVERSE if inverse else _lib.FORWARD)
    return y.view(shape), ld.view(shape)


def unconstrained_rational_quadratic_spline(inputs, unnorm_widths, unnorm_heights, unnorm_derivatives,
                                            inverse=False, lower=-1., upper=1., left=None, right=None,
                                            bottom=None, top=None, min_bin_width=1e-3,
                                            min_bin_height=1e-3, min_derivative=1e-3):
    """(outputs, log-Jacobian diagonal), identity outside the box.  ``unnorm_derivatives`` has
    ``n_bins - 1`` entries (boundary derivatives fixed to 1) or ``n_bins + 1`` (boundary derivatives
    free).  Widths are ``min_bin_width + (1 - min_bin_width * n_bins) * softmax`` (heights alike),
    derivatives ``min_derivative + softplus``; ``min_bin_width * n_bins > 1`` raises ValueError."""
    K = unnorm_widths.shape[-1]
    n_der = unnorm_derivatives.shape[-1]
    if n_der not in (K - 1, K + 1):
        raise ValueError(f'unnorm_derivatives must have n_bins - 1 = {K - 1} or n_bins + 1 = {K + 1} '
                         f'entries, got {n_der}')
    free_edge = n_der == K + 1
    mins = (float(min_bin_width), float(min_bin_height), float(min_derivative))
    has_box = all(v is not None for v in (left, right, bottom, top))
    if has_box and any(torch.is_tensor(v) for v in (left, right, bottom, top)):
        raise NotImplementedError('tensor-valued boxes are not built')
    if not has_box:
        left = bottom = lower
        right = top = upper
    fmeta = [float(lower), float(upper), float(left), float(right), float(bottom), float(top)]
    if free_edge or mins != RQS_DEFAULTS:
        fmeta += [1., *mins, float(free_edge), 0., 0.]
    return _row_params_call(_lib.RQS, inputs, [unnorm_widths, unnorm_heights, unnorm_derivatives], K,
                            inverse, fmeta, has_box)


def unconstrained_cubic_spline(inputs, unnormalized_widths, unnormalized_heights, unnorm_derivatives,
                               inverse=False, lower=-1, upper=1, tails='linear', min_bin_width=1e-2,
                               min_bin_height=1e-2, eps=1e-5, quadratic_threshold=1e-3):
    if tails != 'linear':
        raise RuntimeError('{} tails are not implemented.'.format(tails))
    consts = (float(min_bin_width), float(min_bin_height), float(eps), float(quadratic_threshold))
    K = unnormalized_widths.shape[-1]
    fmeta = [float(lower), float(upper)] * 3
    if consts != CUBIC_DEFAULTS:
        fmeta += [1., consts[0], consts[1], 0., 0., consts[2], consts[3]]
    return _row_params_call(_lib.CUBIC, inputs, [unnormalized_widths, unnormalized_heights,
                                                 unnorm_derivatives], K, inverse, fmeta, False)
