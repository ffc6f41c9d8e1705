"""byteps_b200.torch - the user-facing API (drop-in for ``byteps.torch``).

Parity: /root/reference/byteps/torch/__init__.py:23-466.  Same entry points:
``init/shutdown/suspend/resume/rank/size/local_rank/local_size``,
``push_pull[_async][_inplace]``, ``poll/synchronize/declare``,
``DistributedOptimizer``, ``broadcast_parameters/optimizer_state/object``,
``Compression``; ``parallel.DistributedDataParallel`` and
``cross_barrier.CrossBarrier`` live in their sub-modules like in the reference.

What is different underneath: on CUDA the optimizer does not issue one
push_pull per parameter.  Gradients live in a symmetric NVLink-mapped arena and
are exchanged bucket by bucket by one fused sm_100a kernel each
(:mod:`byteps_b200.parallel.bucket`); with ``fused_update=True`` the kernel also
applies the SGD/Adam step on fp32 master weights and all-gathers the new
parameters instead of the gradients.
"""
from __future__ import annotations

import io
import math
import os
from contextlib import contextmanager

import cloudpickle
import torch

from ..common import config as _config
from ..common import engine as _engine
from .compression import Compression
from .ops import (byteps_torch_set_num_grads, declare, get_pushpull_speed, init, local_rank, local_size, poll,
                  push_pull, push_pull_async, push_pull_async_inplace, push_pull_group_sync_inplace,
                  push_pull_inplace, rank, resume, set_learning_rate, shutdown, size, suspend, synchronize)
from .ops import push_pull_async_inplace as byteps_push_pull

__all__ = [
    "init", "shutdown", "suspend", "resume", "rank", "size", "local_rank", "local_size", "get_pushpull_speed",
    "push_pull", "push_pull_async", "push_pull_inplace", "push_pull_async_inplace", "push_pull_group_sync_inplace",
    "poll", "synchronize", "declare", "byteps_torch_set_num_grads", "DistributedOptimizer", "broadcast_parameters",
    "broadcast_optimizer_state", "broadcast_object", "Compression", "set_learning_rate",
]


def _wire_of(compression):
    if compression is Compression.fp16:
        return torch.float16
    if compression is getattr(Compression, "bf16", None):
        return torch.bfloat16
    return None


def _fused_kind(optimizer_cls, param_groups):
    name = optimizer_cls.__name__
    if issubclass(optimizer_cls, torch.optim.SGD):
        return "sgd"
    if issubclass(optimizer_cls, torch.optim.AdamW):
        return "adamw"
    if issubclass(optimizer_cls, torch.optim.Adam):
        if any(g.get("amsgrad", False) for g in param_groups):
            return None
        return "adam"
    del name
    return None


def _check_max_grad_norm(v):
    if v is None:
        return None
    v = float(v)
    if not math.isfinite(v) or v <= 0:
        raise ValueError("max_grad_norm must be a finite number > 0, got %r" % v)
    return v


class _DistributedOptimizer(torch.optim.Optimizer):
    def __init__(self, params, named_parameters, compression, backward_passes_per_step=1, fused_update=None,
                 bucket_bytes=None, compression_params=None, max_grad_norm=None):
        super(self.__class__, self).__init__(params)
        self._compression = compression
        from ..common.compression_params import translate

        self._compress_kwargs = translate(compression_params, self.defaults)
        named_parameters = list(named_parameters) if named_parameters is not None else []
        self._enable_async = (int(os.getenv('BYTEPS_ENABLE_ASYNC', 0)) != 0)
        self._async_seeded = False
        self._max_grad_norm = _check_max_grad_norm(max_grad_norm)
        self._grad_norm = None
        if self._enable_async and self._max_grad_norm is not None:
            raise ValueError("max_grad_norm is not supported with BYTEPS_ENABLE_ASYNC=1: workers push weight deltas, "
                             "there is no averaged gradient to clip")
        if self._enable_async:
            assert int(os.getenv('DMLC_NUM_WORKER', 1)) > 1, "Async is only valid for distributed training"
        if any(not isinstance(p, tuple) for p in named_parameters):
            raise ValueError('named_parameters should be a sequence of tuples (name, parameter), '
                             'usually produced by model.named_parameters().')
        dups = _DistributedOptimizer.find_duplicates([k for k, _ in named_parameters])
        if dups:
            raise ValueError('Parameter names in named_parameters must be unique. '
                             'Found duplicates: %s' % ', '.join(dups))
        all_params = [p for g in self.param_groups for p in g['params']]
        if named_parameters:
            self._parameter_names = {p: n for n, p in named_parameters}
        else:
            self._parameter_names = {p: 'push_pull.noname.%s' % i for i, p in enumerate(all_params)}
        self.backward_passes_per_step = backward_passes_per_step
        self._push_pull_delay = {p: backward_passes_per_step for p in all_params if p.requires_grad}
        self._handles = {}
        self._grad_accs = []
        self._hook_handles = []
        self._requires_update = set()
        self._should_sync = True
        self._sync = None        # BucketedGradSync on the symmetric-memory path
        self._fused = None
        # priority: parameters needed first by the next forward go first
        self._priority = {p: -i for i, p in enumerate(all_params)}

        # declare in sorted-name order, gradients first then parameters, so
        # keys are identical on all ranks (reference: "two loops for load-balancing")
        for name in sorted(self._parameter_names.values()):
            declare("Gradient." + name, **self._compress_kwargs)
        for name in sorted(self._parameter_names.values()):
            declare("Parameter." + name)
        if self._compress_kwargs:
            # error feedback rescales its residual by lr_prev / lr: the compressors must know the rate BEFORE the
            # first exchange, not from the first step() on (the residual of step 1 was scaled by 1 / lr otherwise)
            set_learning_rate(self.param_groups[0]["lr"])

        eng = _engine()
        if fused_update is None:
            fused_update = os.getenv("BYTEPS_FUSED_OPTIMIZER", "0") not in ("0", "")
        on_cuda = all(p.is_cuda for p in all_params) and torch.cuda.is_available()
        # lossy compressors work per tensor (own error-feedback state): they take the per-parameter path
        want_symm = on_cuda and not self._enable_async and not self._compress_kwargs and (
            eng.backend == "symm" or (eng.backend == "local" and fused_update))
        if want_symm:
            from ..parallel.bucket import BucketedGradSync

            kind = _fused_kind(self.__class__.__mro__[1], self.param_groups) if fused_update else None
            if fused_update and kind is None:
                raise ValueError("fused_update supports SGD, Adam and AdamW (no amsgrad)")
            self._fused = kind
            self._sync = BucketedGradSync(eng, self.param_groups, fused=kind, wire_dtype=_wire_of(compression),
                                          bucket_bytes=bucket_bytes,
                                          backward_passes_per_step=backward_passes_per_step,
                                          priority_of=self._priority,
                                          max_grad_norm=self._max_grad_norm if kind else None)
            if kind:
                self._sync.refresh_hparams()
        elif size() > 1 or eng.backend == "ps":
            # one worker behind a server (BYTEPS_FORCE_DISTRIBUTED=1, the reference's test harness) still goes
            # through the servers: that is what applies the two compression stages
            self._register_hooks()

    @staticmethod
    def find_duplicates(lst):
        seen, dups = set(), set()
        for el in lst:
            if el in seen:
                dups.add(el)
            seen.add(el)
        return dups

    def set_backward_passes_per_step(self, passes):
        self.backward_passes_per_step = passes
        for p in self._push_pull_delay:
            self._push_pull_delay[p] = passes
        if self._sync is not None:
            self._sync.set_backward_passes_per_step(passes)

    # ---- generic (per-parameter) path: gloo / nccl / ps transports -------------
    def _register_hooks(self):
        for param_group in self.param_groups:
            for p in param_group['params']:
                if p.requires_grad:
                    if p.grad is None:
                        p.grad = torch.zeros_like(p)
                    self._requires_update.add(p)
                    self._hook_handles.append(p.register_post_accumulate_grad_hook(self._make_hook(p)))

    def _push_pull_grad_async(self, p):
        name = self._parameter_names.get(p)
        if self._enable_async:
            return None, None   # the real handle is created in step()
        if p.grad is None:      # unused this iteration and cleared by zero_grad(set_to_none=True): contribute zeros
            p.grad = torch.zeros_like(p)
        tensor = p.grad
        if not tensor.is_contiguous() and _dense_tensor(tensor):
            # channels_last & co: the sum is elementwise, exchange the dense storage as a flat view
            tensor = torch.as_strided(tensor, (tensor.numel(),), (1,), tensor.storage_offset())
        tensor_compressed, ctx = self._compression.compress(tensor)
        handle = byteps_push_pull(tensor_compressed, average=True, name="Gradient." + name,
                                  priority=self._priority.get(p, 0))
        return handle, (ctx, tensor_compressed)

    def _make_hook(self, p):
        def hook(*ignore):
            if p in self._handles and self._handles[p][0] is not None:
                if self._push_pull_delay[p] <= 0:
                    raise AssertionError(
                        "Gradients were computed more than backward_passes_per_step times before call "
                        "to step(). Increase backward_passes_per_step to accumulate gradients locally.")
            assert not p.grad.requires_grad
            assert self._push_pull_delay[p] > 0
            handle, ctx = None, None
            self._push_pull_delay[p] -= 1
            if self._push_pull_delay[p] == 0:
                handle, ctx = self._push_pull_grad_async(p)
            self._handles[p] = (handle, ctx)
        return hook

    def synchronize(self):
        if self._sync is not None:
            self._sync.synchronize()
            return
        missing_p = self._requires_update - set(self._handles.keys())
        for p in sorted(missing_p, key=lambda q: self._parameter_names.get(q)):
            self._handles[p] = self._push_pull_grad_async(p)
        for p, (handle, ctx) in list(self._handles.items()):
            if handle is None:
                self._handles[p] = self._push_pull_grad_async(p)
        for p, (handle, ctx) in self._handles.items():
            output = synchronize(handle)
            self._push_pull_delay[p] = self.backward_passes_per_step
            if not self._enable_async and ctx is not None:
                cctx, _ = ctx
                tmp = self._compression.decompress(output, cctx)
                if tmp.data_ptr() != p.grad.data_ptr():
                    if tmp.shape != p.grad.shape:   # flat view of a dense, permuted gradient
                        torch.as_strided(p.grad, (p.grad.numel(),), (1,), p.grad.storage_offset()).copy_(tmp)
                    else:
                        p.grad.copy_(tmp)
        self._handles.clear()

    @contextmanager
    def skip_synchronize(self):
        if self._enable_async:
            raise AssertionError("skip_synchronize cannot be used in async training")
        self._should_sync = False
        try:
            yield
        finally:
            self._should_sync = True

    def zero_grad(self, set_to_none=False):
        if self._sync is not None:
            self._sync.zero_grad()      # one memset per bucket; .grad stays an arena view
            return
        return super(self.__class__, self).zero_grad(set_to_none=set_to_none)

    def refresh_hparams(self):
        """Fused mode + CUDA graphs: call before every replay of a captured step
        so lr/momentum/Adam bias corrections of that step reach the kernels
        (eager ``step()`` does the equivalent by itself)."""
        if self._sync is not None:
            self._sync.pre_replay()

    def step(self, closure=None):
        if self._enable_async:
            old_weight_map = {p: p.data.clone().detach() for p in self._handles}
            if not self._async_seeded:
                # the server accumulates deltas ONTO its stored copy: seed it with the weights (in name order, the
                # same on every worker; workers are expected to start from broadcast parameters).  The reference
                # seeds it with whatever the first push_pull of that name carries, i.e. a delta.
                for p in sorted(old_weight_map, key=lambda q: self._parameter_names.get(q)):
                    _engine().init_tensor("AsyncParam." + self._parameter_names.get(p), old_weight_map[p])
                self._async_seeded = True
            loss = super(self.__class__, self).step(closure)
            for p, (h, _) in list(self._handles.items()):
                p.data.sub_(old_weight_map.get(p))   # weight delta, pushed in place
                if h is None:
                    name = self._parameter_names.get(p)
                    handle = byteps_push_pull(p, average=False, name="AsyncParam." + name)
                    self._handles[p] = (handle, None)
            self.synchronize()
            return loss
        if self._fused:
            loss = closure() if closure is not None else None
            # the update already happened inside the exchange kernels
            if self._should_sync:
                self.synchronize()
            self._sync.step_done()
            return loss
        if self._compress_kwargs:
            set_learning_rate(self.param_groups[0]["lr"])     # error feedback rescales by lr_prev/lr
        if self._should_sync:
            self.synchronize()
        if self._max_grad_norm is not None:
            params = [p for g in self.param_groups for p in g["params"] if p.requires_grad]
            self._grad_norm = torch.nn.utils.clip_grad_norm_(params, self._max_grad_norm)
        return super(self.__class__, self).step(closure)

    @property
    def max_grad_norm(self):
        return self._max_grad_norm

    @max_grad_norm.setter
    def max_grad_norm(self, value):
        if value is None or self._max_grad_norm is None:
            raise ValueError("max_grad_norm can be changed, not switched on or off, after construction")
        self._max_grad_norm = _check_max_grad_norm(value)
        if self._fused:
            self._sync.max_grad_norm = self._max_grad_norm
            self._sync.refresh_hparams()      # eager: reaches the next step; graphs: refresh_hparams() before replay

    def grad_norm(self):
        """With ``max_grad_norm``: the total L2 norm of the averaged gradients of the last step, before clipping (what
        ``clip_grad_norm_`` returns), as a 0-dim fp32 tensor.  On the fused path it is one device tensor that every
        step (and CUDA-graph replay) overwrites; reading it does not synchronise.  ``None`` without clipping, or
        before the first step on the other paths."""
        if self._fused and self._sync.clip:
            return self._sync.grad_norm()
        return self._grad_norm

    @property
    def grad_sync(self):
        return self._sync


def DistributedOptimizer(optimizer, named_parameters=None, compression=Compression.none,
                         backward_passes_per_step=1, fused_update=None, bucket_bytes=None, compression_params=None,
                         max_grad_norm=None):
    """Wrap ``optimizer`` so gradients are averaged over all processes before
    ``step()``; communication overlaps with ``loss.backward()``.

    Arguments match the reference (optimizer, named_parameters, compression,
    backward_passes_per_step).  Extras: ``fused_update=True`` applies the
    SGD/Adam(W) step on fp32 master weights inside the exchange kernel;
    ``bucket_bytes`` sets the fusion granularity; ``compression_params`` (e.g.
    ``{"compressor": "topk", "k": 0.01, "ef": "vanilla"}``, docs/gradient-compression.md)
    turns on lossy gradient compression per tensor - GPU kernels over NVLink, or the
    worker/server compressors in CPU-server mode.

    ``max_grad_norm`` (a finite float > 0) clips the averaged gradients of every
    ``step()`` to that global L2 norm before the update, with the semantics of
    ``torch.nn.utils.clip_grad_norm_`` over every parameter that requires grad (one
    without a gradient counts as zero; the norm is of the gradients after the loss
    scale is removed; a NaN/inf norm propagates like in torch).  ``grad_norm()``
    returns the norm before clipping; ``opt.max_grad_norm`` may be changed between
    steps (under ``GraphedStep`` it reaches the kernels through ``refresh_hparams``,
    like ``lr``).  With ``fused_update=True`` the norm is computed on the device
    between the reduction and the update, inside the exchange, with no host
    synchronisation.  After such a step this rank's shard of each bucket in ``p.grad``
    holds the averaged gradient, the rest this rank's local one; as without clipping,
    the gradient buffers are otherwise unspecified after ``step()``.  On every other
    path ``step()`` calls ``clip_grad_norm_`` between ``synchronize()`` and the
    wrapped optimizer's step.  Not available with ``BYTEPS_ENABLE_ASYNC=1`` or with
    ``Compression.fp16/bf16`` on fp32 parameters of the fused path.

    ``synchronize()`` forces completion (e.g. before gradient clipping without
    ``max_grad_norm``; on the fused path it has already applied the update, so clip
    with ``max_grad_norm`` there), ``skip_synchronize()`` lets a following
    ``step()`` skip it.
    """
    cls = type(optimizer.__class__.__name__, (optimizer.__class__,), dict(_DistributedOptimizer.__dict__))
    return cls(optimizer.param_groups, named_parameters, compression, backward_passes_per_step, fused_update,
               bucket_bytes, compression_params, max_grad_norm)


def broadcast_parameters(params, root_rank, prefix="Parameter."):
    """Broadcast parameters from ``root_rank`` (dict such as ``state_dict()``,
    or a list of tensors / (name, tensor) pairs).  Implemented, like the
    reference, as zero-on-non-root followed by a sum push_pull."""
    if isinstance(params, dict):
        params = sorted(params.items())
    elif isinstance(params, list):
        params = [p if isinstance(p, tuple) else (None, p) for p in params]
    else:
        raise ValueError('invalid params of type: %s' % type(params))
    handles = []
    for name, p in params:
        if not torch.is_tensor(p):
            continue
        t = p.detach()
        if not t.is_contiguous():
            # e.g. channels_last weights: exchange the dense storage instead
            if not _dense_tensor(t):
                raise ValueError("cannot broadcast non-dense tensor %s" % name)
            t = torch.as_strided(t, (t.numel(),), (1,), t.storage_offset())
        if rank() != root_rank:
            t.zero_()
        handles.append(byteps_push_pull(t, average=False, name=(prefix + name) if name else None))
    for h in handles:
        synchronize(h)
    from ..parallel.bucket import resync_fused_masters

    resync_fused_masters()


def _dense_tensor(t):
    if t.numel() == 0:
        return True
    span = 1 + sum((s - 1) * st for s, st in zip(t.size(), t.stride()))
    return span == t.numel()


def _materialised_state(optimizer):
    """state_dict of an optimizer whose per-parameter state exists.  A fresh optimizer has none until its first
    step: take one step of the INNER optimizer on zero gradients and undo whatever it did to the weights
    (weight decay moves them even with a zero gradient)."""
    sd = optimizer.state_dict()
    if sd["state"] or getattr(optimizer, "_fused", None):
        return sd
    weights = [p for g in optimizer.param_groups for p in g["params"]]
    for p in weights:
        if p.requires_grad and p.grad is None:
            p.grad = torch.zeros_like(p)
    keep = [p.detach().clone() for p in weights]
    inner = super(optimizer.__class__, optimizer) if hasattr(optimizer, "_push_pull_delay") else optimizer
    inner.step()
    for p, v in zip(weights, keep):
        p.data.copy_(v)
    return optimizer.state_dict()


def broadcast_optimizer_state(optimizer, root_rank, prefix="Parameter."):
    """Make every process's optimizer state equal to ``root_rank``'s: tensor entries (momentum buffers, Adam
    moments, ...) are broadcast in place like parameters, everything else - python / 0-dim state entries such as
    ``step`` and the options of every param group (lr, betas, ...) - travels as one pickled tree.
    (Reference: byteps/torch/__init__.py:302-424.)"""
    if isinstance(optimizer, torch.optim.LBFGS):
        raise ValueError("cannot broadcast torch.optim.LBFGS state")
    sd = _materialised_state(optimizer)
    if not sd["state"]:
        return
    tensors = []                                     # (name, tensor); names are equal on all ranks by construction
    plain = {"groups": [{k: v for k, v in g.items() if k != "params"} for g in sd["param_groups"]], "state": {}}
    for g in sd["param_groups"]:
        for pid in g["params"]:
            for field, val in sd["state"].get(pid, {}).items():
                if torch.is_tensor(val) and val.dim() > 0 and val.numel() > 0:
                    tensors.append(("%s.%s" % (field, pid), val))
                else:
                    plain["state"].setdefault(pid, {})[field] = val
    broadcast_parameters(tensors, root_rank, prefix)
    plain = broadcast_object(plain, root_rank, name="optimizer_state.plain")
    for live, stored, opts in zip(optimizer.param_groups, sd["param_groups"], plain["groups"]):
        live.update(opts)
        stored.update(opts)             # load_state_dict below must not put the old options back
    for pid, fields in plain["state"].items():
        sd["state"][pid].update(fields)
    # tensors were overwritten in place; the plain entries reach the optimizer through load_state_dict (torch
    # casts a python `step` back to the tensor form the optimizer keeps)
    optimizer.load_state_dict(sd)


def broadcast_object(obj, root_rank=0, name=None):
    """Pickle ``obj`` on ``root_rank`` and return it on every process."""
    if name is None:
        name = type(obj).__name__
    if rank() == root_rank:
        b = io.BytesIO()
        cloudpickle.dump(obj, b)
        t = torch.frombuffer(bytearray(b.getvalue()), dtype=torch.uint8).clone()
        sz = torch.tensor([t.shape[0]], dtype=torch.int32)
        broadcast_parameters([(name + '.sz', sz)], root_rank, prefix="Size.")
    else:
        sz = torch.tensor([0], dtype=torch.int32)
        broadcast_parameters([(name + '.sz', sz)], root_rank, prefix="Size.")
        t = torch.zeros(int(sz.item()), dtype=torch.uint8)
    broadcast_parameters([(name + '.t', t)], root_rank, prefix="Parameter.")
    if rank() != root_rank:
        obj = cloudpickle.load(io.BytesIO(t.numpy().tobytes()))
    return obj
