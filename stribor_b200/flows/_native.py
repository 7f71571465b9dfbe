"""Shared host-side description of a fused layer (see _ops.py for the wire format)."""
from __future__ import annotations

import ctypes as C
import os

import torch

from .. import _epoch, _lib, _ops
from ..net.mlp import MLP


def net_meta(net):
    """-> (dims, act, final_act, params) for an MLP conditioner, or raise NotImplementedError."""
    if not isinstance(net, MLP):
        raise NotImplementedError(
            f'latent_net of type {type(net).__name__} is not fused; use stribor_b200.net.MLP')
    return net.describe()


def build_meta(kind, dim, latent_dim, cond_x, time_input, n_bins, inv_own, zero_cond, net, n_extra,
               has_box=0, mask_list=None):
    if net is None:
        dims, act, fact, params = [], 0, 0, None
        n_linear = 0
    else:
        dims, act, fact, params = net_meta(net)
        n_linear = len(dims) - 1
    n_params = (2 * n_linear if n_linear else 1) + n_extra
    meta = [kind, dim, latent_dim, int(cond_x), int(time_input), n_bins, int(inv_own), int(zero_cond),
            act, fact, n_linear, n_params, int(has_box), 0] + list(dims)
    if cond_x:
        assert mask_list is not None and len(mask_list) == dim
        meta += [int(v) for v in mask_list]
    return meta, params


class PackedCache:
    """Device image of a layer's weights for the tcgen05 kernel, rebuilt when they change.

    "Change" is detected through the parameters' storage pointers and autograd version counters, which every
    in-place op on the parameter itself bumps (optimizer steps, ``load_state_dict``, ``p.mul_()`` under
    ``no_grad``).  Writes through ``p.data`` (``p.data.copy_(ema)``, ``p.data.mul_()``) bypass the counter:
    after those call ``stribor_b200.invalidate_packed(module)`` (the owning layers also invalidate on
    ``.to()/.cuda()``, ``train()/eval()`` and ``load_state_dict``)."""

    def __init__(self):
        self.key = None
        self.buf = None
        self.event = None
        self.seen = set()

    def invalidate(self):
        self.key = None
        _epoch.bump()                 # cached call plans hold the image (flow.run_chain)

    def order_after_pack(self, stream):
        """A cached plan is about to read the image on ``stream``."""
        if self.buf is not None and stream.cuda_stream not in self.seen:
            stream.wait_event(self.event)
            self.seen.add(stream.cuda_stream)

    def get(self, meta, fmeta, mask, params):
        if not params or not params[0].is_cuda or os.environ.get('STRIBOR_B200_FORCE_GENERIC') == '1':
            return None
        if params[0].dtype != torch.float32:
            return None               # float64 layers run on the CUDA-core kernels only: no image
        key = (tuple(meta), tuple(fmeta), tuple((p.data_ptr(), p._version) for p in params))
        if key == self.key:
            if self.buf is not None:
                cur = torch.cuda.current_stream(self.buf.device)
                if cur.cuda_stream not in self.seen:      # first use from another stream: order it after the pack
                    cur.wait_event(self.event)
                    self.seen.add(cur.cuda_stream)
            return self.buf
        lib = _lib.lib()
        detached = [p.detach() for p in params]
        L = _ops.make_struct(meta, fmeta, mask, detached, None)
        nbytes = int(lib.stb_packed_bytes(C.byref(L)))
        buf = None
        if nbytes > 0:
            buf = torch.empty(nbytes, dtype=torch.uint8, device=params[0].device)
            with torch.cuda.device(buf.device):
                stream = torch.cuda.current_stream(buf.device)
                _lib.check(lib.stb_pack_layer(C.byref(L), buf.data_ptr(), stream.cuda_stream))
                # the image may be consumed from OTHER streams next: they wait on this event at their first
                # use (no host synchronisation -- the training step repacks every layer after each update)
                self.event = torch.cuda.Event()
                self.event.record(stream)
                self.seen = {stream.cuda_stream}
        self.key, self.buf = key, buf
        return buf


def device_mask(cache, mask_func, dim, device):
    """(uint8 [dim] mask on `device`, the same mask as a python list), cached per (dim, device)."""
    k = (dim, str(device))
    if k not in cache:
        if ('host', dim) not in cache:
            m = mask_func(dim)
            if m.numel() == 1 and dim != 1:
                m = m.expand(dim)
            cache[('host', dim)] = (m != 0).to(torch.uint8).contiguous()
        host = cache[('host', dim)]
        cache[k] = (host.to(device), host.tolist())
    return cache[k]


def fusable(net) -> bool:
    """Can the kernels evaluate this conditioner themselves?"""
    if not isinstance(net, MLP) or type(net).forward is not MLP.forward:
        return False                  # (a subclass that overrides forward is evaluated as the module it is)
    try:
        net.describe()
        return True
    except NotImplementedError:
        return False


def needs_autograd(module, *tensors) -> bool:
    """True when a gradient could flow through this call (parameters or inputs require grad)."""
    if not torch.is_grad_enabled():
        return False
    if any(t is not None and t.requires_grad for t in tensors):
        return True
    return any(p.requires_grad for p in module.parameters())


def row_params_from_net(net, z, rows_idx=None):
    """Evaluate a conditioner as a PyTorch module (training path, or a conditioner the kernels do
    not fuse).  For an ``MLP`` with ``rows_idx`` only those rows of the LAST Linear are evaluated (the
    transformed dims' parameters, "masked minimum"); any other module is simply called."""
    if not isinstance(net, MLP) or net._wrapped or type(net).forward is not MLP.forward:
        out = net(z)
        return out if rows_idx is None else out.index_select(-1, rows_idx)
    mods = list(net.net)
    last = max(i for i, m in enumerate(mods) if isinstance(m, torch.nn.Linear))
    h = z
    for m in mods[:last]:
        h = m(h)
    lin = mods[last]
    if rows_idx is None:
        out = torch.nn.functional.linear(h, lin.weight, lin.bias)
    else:
        out = torch.nn.functional.linear(h, lin.weight.index_select(0, rows_idx), lin.bias.index_select(0, rows_idx))
    for m in mods[last + 1:]:
        out = m(out)
    return out


class PackedOwner:
    """Mixin of the layers that own a ``PackedCache`` (``self._packed``): drop the image whenever the module's
    tensors are moved / cast, its mode switches or a state dict is loaded."""

    def invalidate_packed(self):
        self._packed.invalidate()

    def _apply(self, fn, *args, **kwargs):
        self._packed.invalidate()
        return super()._apply(fn, *args, **kwargs)

    def train(self, mode: bool = True):
        self._packed.invalidate()
        return super().train(mode)

    def _load_from_state_dict(self, *args, **kwargs):
        self._packed.invalidate()
        return super()._load_from_state_dict(*args, **kwargs)


def invalidate_packed(module: torch.nn.Module):
    """Drop every cached tensor-core weight image under ``module``; the next call repacks from the live
    weights.  Needed only after writes that bypass autograd's version counter (``p.data.<op>_()``)."""
    for m in module.modules():
        if isinstance(m, PackedOwner):
            m.invalidate_packed()


_LAYER_API = ('forward', 'inverse', 'log_det_jacobian', 'forward_and_log_det_jacobian', 'inverse_and_log_det_jacobian')


def layer_is_plain(layer) -> bool:
    """Does ``layer`` behave as the class of THIS package it derives from?  A user subclass that overrides one of the
    transform methods (say, a coupling that perturbs its input) must not be replaced by the fused whole-chain call,
    which talks to the kernels directly: compare the methods with those of the nearest package class in the MRO."""
    cls = type(layer)
    base = next((c for c in cls.__mro__ if c.__module__.startswith('stribor_b200')), None)
    return base is not None and all(getattr(cls, n, None) is getattr(base, n, None) for n in _LAYER_API)
