"""Half-precision training with fp32 master weights.

Parity: /root/reference/byteps/misc/imagenet18/__init__.py:39-382
(``DistributedOptimizer`` for fp16 models: fp16 params + fp32 master copy,
gradients pushed with priority = order of first appearance, per-parameter SGD
on the master as each handle completes, copy back to fp16, static/dynamic loss
scale).  On B200 this is the *default shape* of the fused path: the exchange
kernel reads bf16/fp16 gradients, accumulates in fp32, divides by
loss_scale*size, updates the fp32 master shard and writes the half-precision
weights to every rank - all in one kernel per bucket.
"""
from __future__ import annotations

import torch

from . import DistributedOptimizer, _check_max_grad_norm


class HalfPrecisionDistributedOptimizer:
    """``loss_scale`` static: fused path (everything inside the exchange kernels).
    ``dynamic_loss_scale=True``: the step must be skippable after the reduced gradients have been
    inspected, so the exchange and the update are separate - gradients are averaged by the bucketed
    (or per-parameter) exchange, checked for inf/nan, unscaled into fp32 master gradients, the wrapped
    optimizer steps on fp32 MASTER copies and the half-precision weights are refreshed from them; the
    scale halves on overflow (step skipped) and doubles after ``scale_window`` clean steps."""

    def __init__(self, optimizer, named_parameters=None, loss_scale: float = 1.0, dynamic_loss_scale: bool = False,
                 scale_window: int = 1000, bucket_bytes=None, max_grad_norm=None):
        self.loss_scale = float(loss_scale)
        self.dynamic = bool(dynamic_loss_scale)
        self.scale_window = int(scale_window)
        self._good_steps = 0
        self.skipped_steps = 0
        self._masters = None
        if self.dynamic:
            # the fp32 master gradients are clipped after unscaling, in _dynamic_step
            self._max_grad_norm = _check_max_grad_norm(max_grad_norm)
            self._grad_norm = None
            named = list(named_parameters) if named_parameters is not None else None
            self._opt = DistributedOptimizer(optimizer, named_parameters=named, fused_update=False,
                                             bucket_bytes=bucket_bytes)
            # re-point the optimizer at fp32 master copies (model parameters keep their half dtype)
            self._masters = {}
            for g in self._opt.param_groups:
                half = list(g["params"])
                g["_half_params"] = half
                masters = []
                for p in half:
                    m = p.detach().float().clone().requires_grad_(p.requires_grad)
                    self._masters[p] = m
                    masters.append(m)
                g["params"] = masters
            self._sync = self._opt.grad_sync
            return
        # static scale: the clipped norm is of the unscaled gradients because the kernels fold 1/loss_scale into it
        self._opt = DistributedOptimizer(optimizer, named_parameters=named_parameters, fused_update=True,
                                         bucket_bytes=bucket_bytes, max_grad_norm=max_grad_norm)
        self._sync = self._opt.grad_sync
        if self._sync is not None:
            self._sync.loss_scale = self.loss_scale
            self._sync.refresh_hparams()

    def __getattr__(self, item):
        return getattr(self._opt, item)

    def scale_loss(self, loss):
        return loss * self.loss_scale

    def backward(self, loss):
        self.scale_loss(loss).backward()

    def zero_grad(self, set_to_none=False):
        if self._masters is not None:
            if self._sync is not None:
                self._sync.zero_grad()
            else:
                for p in self._masters:
                    if p.grad is not None:
                        p.grad.zero_()
            return
        self._opt.zero_grad()

    def _dynamic_step(self, closure):
        loss = closure() if closure is not None else None
        self._opt.synchronize()                       # gradients are global averages now (still scaled)
        halves = [p for p in self._masters if p.grad is not None]
        bad = torch.zeros((), device=halves[0].device)
        for p in halves:
            bad = bad + (~torch.isfinite(p.grad)).any().float()
        if bool(bad.item() > 0):                      # identical on every rank: they hold the same averages
            self.loss_scale = max(self.loss_scale / 2.0, 1.0)
            self._good_steps = 0
            self.skipped_steps += 1
            return loss
        inv = 1.0 / self.loss_scale
        for p in halves:
            m = self._masters[p]
            m.grad = p.grad.detach().float().mul_(inv)
        if self._max_grad_norm is not None:
            masters = [m for g in self._opt.param_groups for m in g["params"] if m.requires_grad]
            self._grad_norm = torch.nn.utils.clip_grad_norm_(masters, self._max_grad_norm)
        # the wrapped optimizer's own update (on the masters), bypassing the distributed step's second sync
        type(self._opt).__mro__[1].step(self._opt)
        with torch.no_grad():
            for p in halves:
                p.copy_(self._masters[p])
        self._good_steps += 1
        if self._good_steps % self.scale_window == 0:
            self.loss_scale *= 2.0
        return loss

    def step(self, closure=None):
        if self._masters is not None:
            return self._dynamic_step(closure)
        if self._sync is not None and self._sync.loss_scale != self.loss_scale:
            self._sync.loss_scale = self.loss_scale
            self._sync.refresh_hparams()
        return self._opt.step(closure)

    @property
    def max_grad_norm(self):
        return self._max_grad_norm if self._masters is not None else self._opt.max_grad_norm

    @max_grad_norm.setter
    def max_grad_norm(self, value):
        if self._masters is None:
            self._opt.max_grad_norm = value       # static scale: the fused exchange reads it
            return
        if value is None or self._max_grad_norm is None:
            raise ValueError("max_grad_norm can be changed, not switched on or off, after construction")
        self._max_grad_norm = _check_max_grad_norm(value)

    def grad_norm(self):
        """Total norm of the last step's unscaled, averaged gradients before clipping (``max_grad_norm``)."""
        if self._masters is not None:
            return self._grad_norm
        return self._opt.grad_norm()

    def master_params(self):
        if self._masters is not None:
            return dict(self._masters)
        return self._sync.master_params() if self._sync is not None else {}
