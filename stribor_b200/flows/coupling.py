"""Coupling layers (reference: stribor/flows/coupling.py).

``Coupling`` (coupling.py:10-95): a mask splits the coordinates; the masked part (plus an
optional ``latent``) feeds ``transform.latent_net`` whose output parametrises the element-wise
``transform`` (``Affine`` or ``Spline``) applied to the other part.  Gather, conditioner MLP,
transform and the per-row log|det J| reduction run in ONE kernel per layer.

``ContinuousAffineCoupling`` (coupling.py:98-213): affine coupling whose log-scale and shift
are multiplied by a time embedding so that t = 0 gives the identity.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

import os

from .. import _lib, _ops
from ..flow import Transform, run_layer
from ..net.time_net import TimeLinear
from ..util.mask import get_mask
from ._native import PackedCache, PackedOwner, build_meta, device_mask, fusable, needs_autograd, row_params_from_net, layer_is_plain
from .affine import Affine
from .spline import Spline

__all__ = ['Coupling', 'ContinuousAffineCoupling']


class Coupling(PackedOwner, Transform):
    """
    Args:
        transform: ``Affine`` or ``Spline`` whose ``latent_net`` maps ``dim (+ latent)`` inputs to the
            transform parameters.
        mask: name from ``stribor_b200.util.mask`` -- `none`, `ordered_right_half` (right half
            conditions, left half is transformed), `ordered_left_half`, `random_half`,
            `parity_even`, `parity_odd`.  If ``dim = 1`` use `none`.
        set_data: the mask selects rows of a set (dim -2) instead of coordinates (coupling.py:49-51).

    ``Affine`` and ``Spline`` transforms run in the fused kernels.  A ``Spline`` subclass that overrides one
    of the reference hooks (``_get_params`` / ``spline`` / ``forward_and_log_diag_jacobian``), or any other
    ``ElementwiseTransform``, is composed exactly as the reference does (coupling.py:69-95): conditioning,
    ``transform(x, latent=z)``, blend, masked sum of ``log_diag_jacobian`` -- around whatever kernels that
    transform itself uses.
    """

    def __init__(self, transform, mask: str, set_data: bool = False, **kwargs):
        super().__init__()
        self.transform = transform
        self.mask_func = get_mask(mask)
        self.mask_name = mask
        self.set_data = set_data
        self._masks = {}
        self._packed = PackedCache()
        # set_data: the mask selects ROWS of a set (dim -2).  Masked-out rows are transformed in all
        # their coordinates with conditioning x*0 (+ latent) -- exactly a 'none'-mask coupling on
        # those rows (coupling.py:49-51,61-78); kept out of the module tree (shared parameters).
        self._rows_layer = [Coupling(transform, 'none')] if set_data else None

    def _fusable_transform(self):
        tr = self.transform
        return (isinstance(tr, Affine) or isinstance(tr, Spline)) and tr.plain()

    def chainable(self):
        if not self._fusable_transform() or not layer_is_plain(self):
            return False
        net = self.transform.latent_net
        return (not self.set_data) and (net is None or fusable(net))

    def _run_reference(self, x, latent, direction, want_ldj):
        """coupling.py:53-95 verbatim in structure, for transforms the kernels do not describe."""
        tr = self.transform
        dim = x.shape[-1]
        mask, _ = device_mask(self._masks, self.mask_func, dim, x.device)
        m = mask.to(x.dtype).expand_as(x)

        def cond(v):
            z = v * m
            if dim == 1:
                z = z * 0
            if latent is not None:
                lat = latent if latent.shape[:-1] == v.shape[:-1] else latent.expand(*v.shape[:-1], latent.shape[-1])
                z = torch.cat([z, lat], -1)
            return z

        if direction == _lib.FORWARD:
            out = tr(x, latent=cond(x)) * (1 - m) + x * m
            point = x
        else:
            out = tr.inverse(x, latent=cond(x)) * (1 - m) + x * m
            point = out
        ldj = None
        if want_ldj:
            ldj = (tr.log_diag_jacobian(point, None, latent=cond(point)) * (1 - m)).sum(-1, keepdim=True)
            if direction == _lib.INVERSE:
                ldj = -ldj
        return out, ldj

    def _run_set(self, x, latent, direction, want_ldj):
        *rest, n, d = x.shape
        m = self.mask_func(n)
        if m.numel() == 1 and n != 1:
            m = m.expand(n)
        sel = (m == 0).nonzero().view(-1).to(x.device)
        y = x.clone()
        ldj = x.new_zeros(*rest, n, 1) if want_ldj else None
        if sel.numel():
            lat = None
            if latent is not None and self.transform.latent_net is not None:
                lat = latent.expand(*rest, n, latent.shape[-1]).index_select(-2, sel)
            out, l = self._rows_layer[0]._run(x.index_select(-2, sel), lat, direction, want_ldj)
            y = y.index_copy(-2, sel, out)
            if want_ldj:
                ldj = ldj.index_copy(-2, sel, l)
        return y, ldj

    def describe(self, dim, latent_dim, device):
        if self.set_data:
            raise NotImplementedError('set_data couplings are applied row-group-wise; not part of fused chains')
        tr = self.transform
        net = tr.latent_net
        mask, mask_list = device_mask(self._masks, self.mask_func, dim, device)
        meta, params = build_meta(tr.kind, dim, latent_dim if net is not None else 0, 1, 0, tr.n_bins,
                                  0, dim == 1, net, 0, mask_list=mask_list)
        if net is None:
            params = [tr.const_out(device) if isinstance(tr, Affine) else tr.const_out()]
        params = list(params)
        fmeta = tr.fmeta()
        packed = self._packed.get(meta, fmeta, mask, params) if net is not None else None
        return {'meta': meta, 'fmeta': fmeta, 'mask': mask, 'params': params, 'packed': packed}

    def _run(self, x, latent, direction, want_ldj):
        if self.set_data:
            return self._run_set(x, latent, direction, want_ldj)
        if not self._fusable_transform():
            return self._run_reference(x, latent, direction, want_ldj)
        lat = latent if self.transform.latent_net is not None else None
        net = self.transform.latent_net
        if net is not None and not fusable(net):
            # a conditioner the kernels do not fuse (any nn.Module works here)
            return self._run_autograd(x, lat, direction, want_ldj)
        if net is not None and needs_autograd(self, x, lat):
            d = self._fused_training_desc(x, lat)
            if d is None:      # conditioner through autograd around the element-wise kernels
                return self._run_autograd(x, lat, direction, want_ldj)
            return run_layer(d, x, lat, None, direction, want_ldj)
        d = self.describe(x.shape[-1], 0 if lat is None else lat.shape[-1], x.device)
        return run_layer(d, x, lat, None, direction, want_ldj)

    def _fused_training_desc(self, x, lat):
        """The layer description when ``stb_layer_backward`` differentiates this layer with its conditioner
        fused (tensor-core path: quadratic spline, 16 bins, MLP[64], dim <= 128), else None."""
        if lat is not None or os.environ.get('STRIBOR_B200_TRAIN_HYBRID') == '1':
            return None
        d = self.describe(x.shape[-1], 0, x.device)
        if d['packed'] is None:
            return None
        key = ('fused_bwd', x.shape[-1], str(x.device), tuple(d['meta']))
        if key not in self._masks:
            L = _ops.make_struct(d['meta'], d['fmeta'], d['mask'], [p.detach() for p in d['params']], d['packed'], x.dtype)
            act_ok = d['meta'][8] in (_lib.ACTIVATIONS['Tanh'], _lib.ACTIVATIONS['Sigmoid'], _lib.ACTIVATIONS['ReLU'])
            self._masks[key] = bool(act_ok and _ops.fused_backward_ok(L))
        return d if self._masks[key] else None

    def _run_autograd(self, x, latent, direction, want_ldj):
        """Training path: the conditioner MLP runs through autograd (cuBLAS GEMMs, only the
        transformed dims' rows of its last Linear); gather, transform and log|det J| and their
        gradients are the element-wise CUDA kernels (``row_out`` mode of the C ABI)."""
        tr = self.transform
        dim = x.shape[-1]
        lead = x.shape[:-1]
        mask, mask_list = device_mask(self._masks, self.mask_func, dim, x.device)
        key = ('rows', dim, str(x.device))
        if key not in self._masks:
            P = tr.params_per_dim()
            tr_dims = [j for j, m in enumerate(mask_list) if m == 0]
            if tr.kind == _lib.AFFINE:
                idx = tr_dims + [dim + j for j in tr_dims]
            else:
                idx = [j * P + p for j in tr_dims for p in range(P)]
            self._masks[key] = (torch.tensor(idx, dtype=torch.long, device=x.device),
                                mask.to(x.dtype))
        rows_idx, mask_f = self._masks[key]
        if rows_idx.numel() == 0:
            # every coordinate passes through (dim == 1, coupling.py:62-63): the reference still evaluates the
            # conditioner and multiplies its result by zero, so its parameters receive zero gradients, not None
            zin = x * 0
            if latent is not None:
                zin = torch.cat([zin, latent if latent.shape[:-1] == lead else latent.expand(*lead, latent.shape[-1])], -1)
            zero = tr.latent_net(zin).sum(-1, keepdim=True) * 0
            return x + zero, (zero if want_ldj else None)
        z = x * mask_f
        if dim == 1:
            z = z * 0
        if latent is not None:
            lat = latent if latent.shape[:-1] == lead else latent.expand(*lead, latent.shape[-1])
            z = torch.cat([z, lat], -1)
        prm = row_params_from_net(tr.latent_net, z.reshape(-1, z.shape[-1]), rows_idx)
        meta, _ = build_meta(tr.kind, dim, 0, 1, 0, tr.n_bins, 0, 0, None, 0, mask_list=mask_list)
        meta[13] = 2                                  # row_mode: compact per-row parameters
        d = {'meta': meta, 'fmeta': tr.fmeta(), 'mask': mask, 'params': [prm.contiguous()], 'packed': None}
        return run_layer(d, x, None, None, direction, want_ldj)

    def forward(self, x, latent=None, reverse=False, **kwargs):
        return self._run(x, latent, _lib.INVERSE if reverse else _lib.FORWARD, False)[0]

    def inverse(self, y, latent=None, **kwargs):
        return self._run(y, latent, _lib.INVERSE, False)[0]

    def log_det_jacobian(self, x, y=None, latent=None, **kwargs):
        return self._run(x, latent, _lib.FORWARD, True)[1]

    # fused versions of the inherited compositions (flow.py:35-47): same values, one kernel
    def forward_and_log_det_jacobian(self, x, latent=None, **kwargs):
        return self._run(x, latent, _lib.FORWARD, True)

    def inverse_and_log_det_jacobian(self, y, latent=None, **kwargs):
        return self._run(y, latent, _lib.INVERSE, True)


class ContinuousAffineCoupling(PackedOwner, Transform):
    """
    Args:
        latent_net: maps ``[x*mask | latent | t]`` to ``2 * dim`` affine parameters
        time_net: ``TimeLinear`` with ``2 * dim`` outputs
        mask: mask name (see ``Coupling``)
        concatenate_time: whether ``t`` is appended to the network input
    """

    def __init__(self, latent_net: nn.Module, time_net: nn.Module, mask: str,
                 concatenate_time: Optional[bool] = True, **kwargs):
        super().__init__()
        self.latent_net = latent_net
        self.mask_func = get_mask(mask)
        self.mask_name = mask
        self.time_net = time_net
        self.concatenate_time = concatenate_time
        self._masks = {}
        self._packed = PackedCache()

    def _linear_time(self):
        """Is the time embedding exactly ``scale * t``?  (``TimeTanh`` / ``TimeLog`` SUBCLASS ``TimeLinear`` as in the
        reference, and a user subclass may override ``forward``: only the class itself is fused into the kernels.)"""
        return type(self.time_net) is TimeLinear

    def chainable(self):
        return fusable(self.latent_net) and self._linear_time() and layer_is_plain(self)

    def _time_scale(self, dim):
        if not self._linear_time():
            raise NotImplementedError(f'time_net {type(self.time_net).__name__} is not fused; use TimeLinear')
        s = self.time_net.scale
        n = s.shape[-1]
        if n == 2 * dim:
            return s.reshape(-1)
        if n == 2:       # chunk(2) gives [..., 1] halves that broadcast over dim (README.md:94-97)
            return s.reshape(2, 1).expand(2, dim).reshape(-1)
        raise ValueError(f'time_net output size {n} does not match 2 * dim = {2 * dim}')

    def describe(self, dim, latent_dim, device):
        mask, mask_list = device_mask(self._masks, self.mask_func, dim, device)
        meta, params = build_meta(_lib.CONT_AFFINE, dim, latent_dim, 1, bool(self.concatenate_time), 0,
                                  0, dim == 1, self.latent_net, 1, mask_list=mask_list)
        params = list(params) + [self._time_scale(dim).contiguous()]
        fmeta = [0., 1.] * 3
        return {'meta': meta, 'fmeta': fmeta, 'mask': mask, 'params': params,
                'packed': self._packed.get(meta, fmeta, mask, params)}

    def _run(self, x, t, latent, direction, want_ldj):
        if t is None:
            raise TypeError('ContinuousAffineCoupling needs the time input `t`')
        if needs_autograd(self, x, t, latent) or not fusable(self.latent_net) or not self._linear_time():
            return self._run_autograd(x, t, latent, direction, want_ldj)
        d = self.describe(x.shape[-1], 0 if latent is None else latent.shape[-1], x.device)
        return run_layer(d, x, latent, t, direction, want_ldj)

    def _run_autograd(self, x, t, latent, direction, want_ldj):
        """Training path: conditioner and time embedding through autograd; the effective affine
        parameters  a = log_scale * t_log_scale,  b = shift * t_shift  (coupling.py:199-205) are handed
        per row to the affine element-wise kernels (forward and backward)."""
        dim = x.shape[-1]
        lead = x.shape[:-1]
        mask, mask_list = device_mask(self._masks, self.mask_func, dim, x.device)
        key = ('rows', dim, str(x.device))
        if key not in self._masks:
            tr_dims = [j for j, m in enumerate(mask_list) if m == 0]
            self._masks[key] = (torch.tensor(tr_dims, dtype=torch.long, device=x.device), mask.to(x.dtype))
        tr_idx, mask_f = self._masks[key]
        if tr_idx.numel() == 0:
            # nothing is transformed (dim == 1): zero -- not None -- gradients for both networks, as the
            # reference's multiply-by-(1 - mask) gives
            zin = x * 0
            if latent is not None:
                zin = torch.cat([zin, latent if latent.shape[:-1] == lead else latent.expand(*lead, latent.shape[-1])], -1)
            tt = t if t.shape[:-1] == lead else t.expand(*lead, 1)
            if self.concatenate_time:
                zin = torch.cat([zin, tt], -1)
            zero = (self.latent_net(zin).sum(-1, keepdim=True) + self.time_net(tt).sum(-1, keepdim=True)) * 0
            return x + zero, (zero if want_ldj else None)
        z = x * mask_f
        if dim == 1:
            z = z * 0
        if latent is not None:
            z = torch.cat([z, latent if latent.shape[:-1] == lead else latent.expand(*lead, latent.shape[-1])], -1)
        tt = t if t.shape[:-1] == lead else t.expand(*lead, 1)
        if self.concatenate_time:
            z = torch.cat([z, tt], -1)
        out = self.latent_net(z.reshape(-1, z.shape[-1]))
        tn = self.time_net(tt.reshape(-1, 1))                    # any time embedding (net/time_net.py)
        ls, sh = out.chunk(2, dim=-1)
        tls, tsh = tn.chunk(2, dim=-1)                           # [rows, dim] or broadcastable [rows, 1]
        a = (ls * tls).index_select(1, tr_idx)
        b = (sh * tsh).index_select(1, tr_idx)
        prm = torch.cat([a, b], -1).contiguous()
        meta, _ = build_meta(_lib.AFFINE, dim, 0, 1, 0, 0, 0, 0, None, 0, mask_list=mask_list)
        meta[13] = 2
        d = {'meta': meta, 'fmeta': [0., 1.] * 3, 'mask': mask, 'params': [prm], 'packed': None}
        return run_layer(d, x, None, None, direction, want_ldj)

    def forward(self, x, t=None, latent=None, **kwargs):
        return self._run(x, t, latent, _lib.FORWARD, False)[0]

    def inverse(self, y, t=None, latent=None, **kwargs):
        return self._run(y, t, latent, _lib.INVERSE, False)[0]

    def log_det_jacobian(self, x, y=None, *, t=None, latent=None, **kwargs):
        return self._run(x, t, latent, _lib.FORWARD, True)[1]

    def forward_and_log_det_jacobian(self, x, t=None, latent=None, *, reverse=False, **kwargs):
        if reverse:      # coupling.py:188-209: the inverse map together with the FORWARD log-det
            y, ldj = self._run(x, t, latent, _lib.INVERSE, True)
            return y, -ldj
        return self._run(x, t, latent, _lib.FORWARD, True)

    def inverse_and_log_det_jacobian(self, y, t=None, latent=None, **kwargs):
        return self._run(y, t, latent, _lib.INVERSE, True)
