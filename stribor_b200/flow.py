"""Transform ABCs and flow containers (reference: stribor/flow.py).

``NormalizingFlow`` keeps the reference API (``forward / inverse / *_and_log_det_jacobian /
log_prob / sample / rsample / log_det_jacobian``, flow.py:90-152).  When every transform is one
of this package's fused layers and no gradient is required, a whole pass is ONE call into the
C ABI (``stb_flow_apply`` / ``stb_flow_log_prob``): the layer loop, the running log|det J| and
the UnitNormal term all stay on the device.  Otherwise it falls back to the reference's
layer-by-layer composition of the same fused per-layer ops, which is differentiable.
"""
from __future__ import annotations

from abc import ABCMeta, abstractmethod
from typing import List, Optional, Tuple, Union

import torch
import torch.nn as nn

import os
import weakref

from . import _epoch, _ops
from .dist.normal import UnitNormal

__all__ = ['Transform', 'ElementwiseTransform', 'NormalizingFlow', 'NeuralFlow']


class Transform(_epoch.Tracked, nn.Module, metaclass=ABCMeta):
    """flow.py:8-47.  Default pair methods compose forward/inverse with ``log_det_jacobian``:
    the inverse's log-det is MINUS the forward log-det evaluated at the recovered input."""

    @abstractmethod
    def forward(self, x, **kwargs):
        pass

    @abstractmethod
    def inverse(self, y, **kwargs):
        pass

    @abstractmethod
    def log_det_jacobian(self, x, y, **kwargs):
        pass

    def jacobian(self, x, y, **kwargs):
        raise NotImplementedError

    def forward_and_log_det_jacobian(self, x, **kwargs):
        y = self.forward(x, **kwargs)
        return y, self.log_det_jacobian(x, y, **kwargs)

    def inverse_and_log_det_jacobian(self, y, **kwargs):
        x = self.inverse(y, **kwargs)
        return x, -self.log_det_jacobian(x, y, **kwargs)


class ElementwiseTransform(Transform):
    """flow.py:50-69."""

    @abstractmethod
    def log_diag_jacobian(self, x, y, **kwargs):
        pass

    def forward_and_log_diag_jacobian(self, x, **kwargs):
        y = self.forward(x, **kwargs)
        return y, self.log_diag_jacobian(x, y, **kwargs)

    def inverse_and_log_diag_jacobian(self, y, **kwargs):
        x = self.inverse(y, **kwargs)
        return x, -self.log_diag_jacobian(x, y, **kwargs)


# --------------------------------------------------------------------------------------------
# helpers shared by the fused layers
# --------------------------------------------------------------------------------------------
def _flat(v: Optional[torch.Tensor], lead, width=None):
    if v is None:
        return None
    if v.shape[:-1] != tuple(lead):
        v = v.expand(*lead, v.shape[-1])
    return v.reshape(-1, v.shape[-1]).contiguous()


def run_layer(desc, x, latent, t, direction, want_ldj):
    """Apply one described layer to x [..., dim] -> (y [..., dim], ldj [..., 1] or None)."""
    lead, dim = x.shape[:-1], x.shape[-1]
    latent, t = _flat(latent, lead), _flat(t, lead)
    _ops.check_layer_tensors(x, latent, t, desc['mask'], desc['params'], desc.get('packed'),
                             int_params=desc['meta'][0] == _ops._lib.PERMUTE)
    y, ldj = _ops.layer_apply(x.reshape(-1, dim).contiguous(), latent, t,
                              desc['mask'], desc['params'], desc.get('packed'), desc['meta'],
                              desc['fmeta'], direction, want_ldj, False)
    return y.view(*lead, dim), (ldj.view(*lead, 1) if want_ldj else None)


def run_layer_diag(desc, x, latent, t, direction):
    lead, dim = x.shape[:-1], x.shape[-1]
    latent, t = _flat(latent, lead), _flat(t, lead)
    _ops.check_layer_tensors(x, latent, t, desc['mask'], desc['params'])
    y, ld = _ops.layer_apply_diag(x.reshape(-1, dim).contiguous(), latent, t,
                                  desc['mask'], desc['params'], desc['meta'], desc['fmeta'], direction)
    return y.view(*lead, dim), ld.view(*lead, dim)


# ---- cached call plans ---------------------------------------------------------------------------------------
# Describing a chain (per layer: mask, weight tensors, packed image, wire-format lists, the ctypes stb_layer) costs
# ~40 us of Python per layer -- more than the GPU spends on a small batch.  The result is kept per ModuleList for as
# long as (1) the structure epoch (_epoch.py) and (2) every parameter's (data_ptr, _version, requires_grad) stand
# still; weak keys, so flows stay picklable / deep-copyable and nothing outlives them.
_records = weakref.WeakKeyDictionary()


class _Record:
    __slots__ = ('epoch', 'plist', 'chainable', 'plans', 'token', 'any_grad')

    def __init__(self, transforms):
        self.epoch = _epoch.value
        self.plist = list(transforms.parameters())
        self.chainable = len(transforms) > 0 and all(hasattr(f, 'chainable') and f.chainable() for f in transforms)
        self.plans = {}
        self.token = None
        self.any_grad = False

    def refresh(self):
        """Re-read the parameters' state; plans built against an older state are dropped."""
        token = tuple([(p.data_ptr(), p._version, p.requires_grad) for p in self.plist])
        if token != self.token:
            self.token = token
            self.any_grad = any(k[2] for k in token)
            self.plans.clear()


def _record(transforms) -> _Record:
    rec = _records.get(transforms)
    if rec is None or rec.epoch != _epoch.value:
        rec = _Record(transforms)            # (constructing it may describe layers; it never moves the epoch itself)
        _records[transforms] = rec
    rec.refresh()
    return rec


def _chain_ok(transforms, tensors) -> bool:
    """Fused whole-chain path: every layer describable, nothing asks for gradients."""
    rec = _record(transforms)
    if not rec.chainable:
        return False                  # foreign modules, un-fused conditioners, set_data couplings:
                                      # layer-by-layer path
    if torch.is_grad_enabled():
        if rec.any_grad or any(v is not None and v.requires_grad for v in tensors):
            return False
    return True


class _Plan:
    __slots__ = ('masks', 'params', 'packed', 'meta', 'fmeta', 'arr', 'keep', 'caches', 'n')


def _build_plan(transforms, dim, latent_dim, x, latent, t) -> _Plan:
    pl = _Plan()
    pl.masks, pl.params, pl.packed, pl.meta, pl.fmeta, pl.caches = [], [], [], [], [], []
    for f in transforms:
        d = f.describe(dim, latent_dim, x.device)
        _ops.check_layer_tensors(x, latent, t, d['mask'], d['params'], d.get('packed'),
                                 int_params=d['meta'][0] == _ops._lib.PERMUTE)
        pl.masks.append(d['mask'] if d['mask'] is not None else x.new_empty(0, dtype=torch.uint8))
        pl.params += [p.detach() for p in d['params']]
        pl.packed.append(d['packed'] if d.get('packed') is not None else x.new_empty(0, dtype=torch.uint8))
        pl.meta += d['meta']
        pl.fmeta += d['fmeta']
        if getattr(f, '_packed', None) is not None:
            pl.caches.append(f._packed)
    pl.arr, pl.keep = _ops.build_layer_array(pl.masks, pl.params, pl.packed, pl.meta, pl.fmeta, x.dtype)
    pl.n = len(pl.masks)
    return pl


def run_chain(transforms, mode, x, latent=None, t=None, want_ldj=False):
    _ops._check_cuda(x, 'input')
    lead, dim = x.shape[:-1], x.shape[-1]
    latent_dim = 0 if latent is None else latent.shape[-1]
    latent, t = _flat(latent, lead), _flat(t, lead)
    rec = _record(transforms)
    # (x.dtype: a plan's layers carry its dtype; an input of the other dtype builds -- and dtype-checks -- its own)
    key = (dim, latent_dim, x.device, x.dtype, os.environ.get('STRIBOR_B200_FORCE_GENERIC'))
    epoch = _epoch.value
    plan = rec.plans.get(key)
    if plan is None:
        plan = _build_plan(transforms, dim, latent_dim, x, latent, t)
        if _epoch.value == epoch:            # describing a layer for the first time may itself move the epoch
            rec.plans[key] = plan
    else:
        # the per-layer checks ran when the plan was built; the call's own tensors are checked every time
        _ops.check_layer_tensors(x, latent, t, None, ())
        if plan.caches:
            cur = torch.cuda.current_stream(x.device)
            for c in plan.caches:
                c.order_after_pack(cur)
    x2 = x.reshape(-1, dim).contiguous()
    if torch.compiler.is_compiling():
        out, vec = _ops.flow_chain(x2, latent, t, plan.masks, plan.params, plan.packed, plan.meta, plan.fmeta, mode, want_ldj)
    else:
        out, vec = _ops.flow_chain_launch(plan.arr, plan.n, x2, latent, t, mode, want_ldj)
    out = out.view(*lead, dim) if out.shape[0] == x.numel() // dim else None      # LOG_PROB_ONLY: no latent rows
    if want_ldj or mode in (_ops.CHAIN_LOG_PROB, _ops.CHAIN_LOG_PROB_ONLY):
        return out, vec.view(*lead, 1)
    return out, None


class NormalizingFlow(Transform):
    """Normalizing flow for density estimation and sampling (flow.py:72-152).

    Args:
        base_dist: base distribution (``UnitNormal`` is fused into the kernels)
        transforms: list of invertible transformations, applied first-to-last by ``forward``
    """

    def __init__(self, base_dist, transforms: List[Transform]):
        super().__init__()
        self.base_dist = base_dist
        self.transforms = nn.ModuleList(transforms)

    # -- chained application ------------------------------------------------------------------
    def _fused(self, x, kwargs):
        extra = set(kwargs) - {'latent', 't'}
        return (not extra) and _chain_ok(self.transforms, (x, kwargs.get('latent'), kwargs.get('t')))

    def forward(self, x, **kwargs):
        if self._fused(x, kwargs):
            return run_chain(self.transforms, _ops.CHAIN_FORWARD, x, kwargs.get('latent'), kwargs.get('t'))[0]
        for f in self.transforms:
            x = f(x, **kwargs)
        return x

    def inverse(self, y, **kwargs):
        if self._fused(y, kwargs):
            return run_chain(self.transforms, _ops.CHAIN_INVERSE, y, kwargs.get('latent'), kwargs.get('t'))[0]
        for f in reversed(self.transforms):
            y = f.inverse(y, **kwargs)
        return y

    def forward_and_log_det_jacobian(self, x, **kwargs):
        if self._fused(x, kwargs):
            return run_chain(self.transforms, _ops.CHAIN_FORWARD, x, kwargs.get('latent'), kwargs.get('t'), True)
        log_det_jac = 0
        for f in self.transforms:
            x, ldj = f.forward_and_log_det_jacobian(x, **kwargs)
            log_det_jac = log_det_jac + ldj
        return x, log_det_jac

    def inverse_and_log_det_jacobian(self, y, **kwargs):
        if self._fused(y, kwargs):
            return run_chain(self.transforms, _ops.CHAIN_INVERSE, y, kwargs.get('latent'), kwargs.get('t'), True)
        log_det_jac = 0
        for f in reversed(self.transforms):
            y, ldj = f.inverse_and_log_det_jacobian(y, **kwargs)
            log_det_jac = log_det_jac + ldj
        return y, log_det_jac

    def log_prob(self, y, **kwargs):
        """flow.py:127-130: base log-density of the inverted point plus the summed log|det J|."""
        if isinstance(self.base_dist, UnitNormal) and self._fused(y, kwargs):
            return run_chain(self.transforms, _ops.CHAIN_LOG_PROB_ONLY, y, kwargs.get('latent'), kwargs.get('t'))[1]
        x, log_det_jac = self.inverse_and_log_det_jacobian(y, **kwargs)
        return self.base_dist.log_prob(x).unsqueeze(-1) + log_det_jac

    def _device(self):
        for p in self.parameters():
            return p.device
        for b in self.buffers():
            return b.device
        return None

    def sample(self, num_samples: Union[Tuple[int], int], *, rsample: bool = False, **kwargs):
        if isinstance(num_samples, int):
            num_samples = (num_samples,)
        draw = self.base_dist.rsample if rsample else self.base_dist.sample
        if isinstance(self.base_dist, UnitNormal):
            x = draw(num_samples, device=self._device())
        else:
            x = draw(num_samples)
        return self.forward(x, **kwargs)

    def rsample(self, num_samples, **kwargs):
        return self.sample(num_samples, **kwargs)          # as the reference: flow.py:145-146

    def log_det_jacobian(self, x, y=None, **kwargs):
        return self.forward_and_log_det_jacobian(x, **kwargs)[1]


class NeuralFlow(nn.Module):
    """Chain of time-conditioned transforms with F(x, t=0) = x (flow.py:155-184)."""

    def __init__(self, transforms: List[Transform]) -> None:
        super().__init__()
        self.transforms = nn.ModuleList(transforms)

    def forward(self, x, t, t0: Optional[torch.Tensor] = None, **kwargs):
        latent = kwargs.get('latent')
        fused = (not (set(kwargs) - {'latent'})) and _chain_ok(self.transforms, (x, t, t0, latent))
        if fused:
            if t0 is not None:
                x = run_chain(self.transforms, _ops.CHAIN_INVERSE, x, latent, t0)[0]
            return run_chain(self.transforms, _ops.CHAIN_FORWARD, x, latent, t)[0]
        if t0 is not None:
            for transform in reversed(self.transforms):
                x = transform.inverse(x, t=t0, **kwargs)
        for transform in self.transforms:
            x = transform(x, t=t, **kwargs)
        return x
