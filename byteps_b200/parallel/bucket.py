"""Zero-copy bucketed gradient synchronisation over symmetric memory.

This is the B200-first replacement for the reference's per-parameter
``push_pull_async_inplace`` hooks (/root/reference/byteps/torch/__init__.py:117-158)
and its per-<=4MB-partition NCCL reduce-scatter/all-gather launches
(core_loops.cc:190-269): gradients LIVE in a peer-mapped arena (``p.grad`` are
strided views into it), buckets are contiguous byte ranges laid out in
backward order, and one fused kernel per bucket does the whole exchange in
place - optionally fused with the fp32 master-weight optimizer step, in which
case the updated parameters (not the gradients) are what is all-gathered.

Everything is stream ordered: a bucket launch waits on an event recorded on the
autograd stream, completion is an event the optimizer step waits on.  No host
thread takes part, so the step can be captured in one CUDA graph.
"""
from __future__ import annotations

import os
import struct
import weakref
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import torch

from ..comm.symm import SymmContext, pick_blocks, wire_code
from ..utils.timing import stamp


def _env_int(name, default):
    v = os.environ.get(name)
    return int(v) if v else default


def _pad8(n: int) -> int:
    return (n + 7) // 8 * 8


def _strided_view(flat: torch.Tensor, p: torch.Tensor, offset: int) -> torch.Tensor:
    """A view of `flat` with p's sizes and strides (keeps channels_last etc.)."""
    if p.is_contiguous():
        return flat[offset:offset + p.numel()].view(p.shape)
    return torch.as_strided(flat, p.size(), p.stride(), offset)


def _dense(p: torch.Tensor) -> bool:
    """True if p's storage footprint equals numel (a permutation of contiguous)."""
    if p.numel() == 0:
        return True
    span = 1 + sum((s - 1) * st for s, st in zip(p.size(), p.stride()))
    return span == p.numel()


@dataclass
class Bucket:
    index: int
    group_index: int
    dtype: torch.dtype
    params: List[torch.nn.Parameter] = field(default_factory=list)
    starts: List[int] = field(default_factory=list)    # element offsets inside the bucket
    numel: int = 0                                     # padded element count (multiple of 8)
    grad_off: int = 0                                  # byte offset of the gradient window in the arena
    param_off: int = -1                                # byte offset of the parameter window (fused mode)
    pending: int = 0
    launched: bool = False
    flat_grad: Optional[torch.Tensor] = None
    flat_param: Optional[torch.Tensor] = None
    master: Optional[torch.Tensor] = None              # fp32 shard
    state0: Optional[torch.Tensor] = None
    state1: Optional[torch.Tensor] = None
    done: Optional[torch.cuda.Event] = None
    priority: int = 0                                  # max priority of the parameters inside (scheduling)
    ring_cls: Optional[tuple] = None                   # (wire code, ring kind) of the ring table it belongs to
    ring_pos: int = -1                                 # position inside that table

    @property
    def nbytes(self) -> int:
        return self.numel * torch.empty((), dtype=self.dtype).element_size()


_LIVE = weakref.WeakSet()


def resync_fused_masters():
    """Re-derive fp32 master shards from the (just broadcast / just loaded)
    parameters of every live fused synchroniser."""
    for s in list(_LIVE):
        if s.fused:
            s.sync_master_from_params()


def clip_update_grid(numels: List[int], itemsize: int, world: int) -> int:
    """CTAs of the clipped update (phase 3) over buckets of `numels` padded elements.  The kernel ends in a barrier
    that pairs the CTAs of equal index across ranks, so the grid must be the same on every rank: it is sized from
    rank 0's shard, the largest (shard_units), not from this rank's, which can be smaller or empty.  Nothing overlaps
    phase 3 (it runs after backward), so it may take two CTAs per SM of a B200 (148 SMs); a fixed cap rather than the
    local device's SM count keeps the grid rank-independent."""
    tiles = 0
    for n in numels:
        groups = n // 8
        per = (groups + world - 1) // world                   # rank 0's shard, in groups of 8 elements
        units = per * 8 * itemsize // 16                      # 16-byte wire units
        tiles += (units + 255) // 256                          # 256 units per tile (kClipTileUnits)
    return max(1, min(tiles, 2 * 148))


_HP_FMT = "<9f3if3i"   # matches csrc/kernels/pushpull.cuh::OptHParams (64 bytes)


class BucketedGradSync:
    """Owns the arena, the buckets and the hooks for one set of parameters."""

    def __init__(self, engine, param_groups, *, fused: Optional[str] = None, wire_dtype: Optional[torch.dtype] = None,
                 bucket_bytes: Optional[int] = None, backward_passes_per_step: int = 1, average: bool = True,
                 priority_of: Optional[Dict] = None, max_grad_norm: Optional[float] = None):
        self.engine = engine
        self.world, self.rank = engine.size, engine.rank
        self.fused = fused                     # None | "sgd" | "adam" | "adamw"
        # global-norm clipping inside the fused exchange (pushpull_clip.cu): phase 1 per bucket from the hooks,
        # norm (phase 2) and clipped update + parameter all-gather (phase 3) from synchronize()
        self.clip = max_grad_norm is not None
        self.max_grad_norm = max_grad_norm
        if self.clip and not fused:
            raise ValueError("max_grad_norm inside the exchange needs a fused optimizer")
        self.average = average
        self.bpps = backward_passes_per_step
        self.bucket_bytes = bucket_bytes or _env_int("BYTEPS_BUCKET_BYTES", 16 << 20)
        self.param_groups = param_groups
        self.wire_override = wire_dtype
        params = [(gi, p) for gi, g in enumerate(param_groups) for p in g["params"] if p.requires_grad]
        if not params:
            raise ValueError("no parameters require gradients")
        if (self.clip and wire_dtype in (torch.bfloat16, torch.float16)
                and any(p.dtype == torch.float32 for _, p in params)):
            raise ValueError("max_grad_norm cannot be combined with a wire cast of fp32 gradients "
                             "(Compression.fp16/bf16): the clipped exchange keeps gradients in the parameter dtype")
        self.device = params[0][1].device
        for _, p in params:
            if p.device != self.device or not p.is_cuda:
                raise ValueError("the symmetric-memory path needs all parameters on one CUDA device")
            if not _dense(p):
                raise ValueError("parameters must be dense (contiguous up to a permutation)")
        # backward order ~ reverse of registration order
        order = list(reversed(params))
        self.buckets: List[Bucket] = []
        open_buckets: Dict = {}       # one open bucket per (param group, dtype)
        for gi, p in order:
            es = p.element_size()
            cur = open_buckets.get((gi, p.dtype))
            if cur is None or ((cur.numel + _pad8(p.numel())) * es > self.bucket_bytes and cur.params):
                cur = Bucket(len(self.buckets), gi, p.dtype)
                self.buckets.append(cur)
                open_buckets[(gi, p.dtype)] = cur
            cur.params.append(p)
            cur.starts.append(cur.numel)
            cur.numel += _pad8(p.numel())
        # ---- arena layout: [grad windows][param windows (fused)][staging (wire cast)][clip norm publish]
        off = 0
        for b in self.buckets:
            b.grad_off = off
            off = (off + b.nbytes + 255) // 256 * 256
        if fused:
            for b in self.buckets:
                b.param_off = off
                off = (off + b.nbytes + 255) // 256 * 256
        self.stage_off = off
        self.stage_bytes = 0
        if self._needs_stage():
            self.stage_bytes = max(self._wire_bytes(b) for b in self.buckets)
            off += (self.stage_bytes + 255) // 256 * 256
        self.clip_pub_off = off
        if self.clip:
            off += 256
        cfg = engine.cfg
        stamp("buckets: layout of %d buckets, arena %d MiB" % (len(self.buckets), off >> 20))
        self.ctx = SymmContext(engine.group, self.device, max(off, 4096), cfg.symm_mode, cfg.use_nvls)
        stamp("buckets: symmetric arena ready")
        if engine.comm_stream is None:
            engine.comm_stream = torch.cuda.Stream(device=self.device, priority=-1)
        self.comm_stream = engine.comm_stream
        self.threads = cfg.comm_threads
        self._param_bucket: Dict[torch.nn.Parameter, Bucket] = {}
        self._delay: Dict[torch.nn.Parameter, int] = {}
        self._grad_views: Dict[torch.nn.Parameter, torch.Tensor] = {}
        for b in self.buckets:
            b.flat_grad = self.ctx.tensor(b.grad_off, b.numel, b.dtype)
            if fused:
                b.flat_param = self.ctx.tensor(b.param_off, b.numel, b.dtype)
            for p, st in zip(b.params, b.starts):
                gv = _strided_view(b.flat_grad, p, st)
                if p.grad is not None:
                    gv.copy_(p.grad)
                p.grad = gv
                self._grad_views[p] = gv
                self._param_bucket[p] = b
                self._delay[p] = self.bpps
                if fused:
                    pv = _strided_view(b.flat_param, p, st)
                    pv.copy_(p.data)
                    p.data = pv
            b.pending = len(b.params)
        if fused:
            self._init_fused_state()
        self._next = 0          # strict mode: next bucket index allowed to launch
        self._strict = os.environ.get("BYTEPS_STRICT_ORDER", "0") not in ("0", "")
        self._hooks = []
        self._step = 0
        self._hp_dirty = True
        self._seg_tables: Dict[int, torch.Tensor] = {}
        self._last_done = None
        self._trace_t0 = None
        self._trace_spans = []
        # which engine moves the NVLink bytes of plain (unfused) buckets:
        #   auto/nvls: multimem.ld_reduce/st when available, else LSU P2P; lsu: force P2P loads/stores;
        #   tma: cp.async.bulk ring; tcgen05: TMA + tensor-core reduction with a TMEM accumulator
        self._reduce_engine = os.environ.get("BYTEPS_REDUCE_ENGINE", "auto").lower()
        # fused optimizer kernels: "tma" streams the fp32 state through shared memory with bulk copies,
        # "lsu" keeps it in registers (also used whenever the gradients need a wire cast)
        self._fused_engine = os.environ.get("BYTEPS_FUSED_ENGINE", "auto").lower()
        if self._fused_engine == "auto":
            # measured in situ (BERT-large AdamW, bench.py): one GPU 23.07 ms/step (tma, 128 CTAs) vs 23.33 (lsu);
            # two GPUs 23.38 vs 23.11 - within noise, so the register kernel (validated on 8 GPUs) stays the
            # multi-GPU default and the TMA kernel (0.92/0.88 vs 0.75/0.77 of the HBM roofline alone) runs solo
            self._fused_engine = "tma" if self.world == 1 else "lsu"
        # CTAs of the TMA variant: its bytes in flight live in shared memory, so a fraction of the SMs
        # saturates HBM/NVLink and the rest stays free for the backward kernels it overlaps with
        self._fused_tma_blocks = _env_int("BYTEPS_FUSED_TMA_BLOCKS", 128)
        self._umma_maps = {}
        self._xlaunches = 0
        self._last_step_launches = 0
        self._priority_of = priority_of or {}
        for b in self.buckets:
            b.priority = max([int(self._priority_of.get(p, 0)) for p in b.params] or [0])
        self._setup_ring()
        self.enabled = True            # DDP.no_sync() turns hooks into local accumulation
        self.auto_finish = None        # DDP: called when every bucket of the iteration was launched
        self._launched = 0
        self._register_hooks()
        _LIVE.add(self)
        torch.cuda.current_stream(self.device).synchronize()
        if self.world > 1:
            engine.group.barrier()
        stamp("buckets: views, fused state, hooks")

    # ------------------------------------------------------------------ layout helpers
    def _wire(self, b: Bucket) -> torch.dtype:
        w = self.wire_override
        if w is not None and b.dtype == torch.float32 and w in (torch.bfloat16, torch.float16):
            return w
        return b.dtype

    def _wire_bytes(self, b: Bucket) -> int:
        return b.numel * torch.empty((), dtype=self._wire(b)).element_size()

    def _needs_stage(self) -> bool:
        return any(self._wire(b) != b.dtype for b in self.buckets)

    def shard_range(self, b: Bucket):
        """Element range [begin, end) of the shard this rank owns in bucket b."""
        units = b.numel // 8
        per = (units + self.world - 1) // self.world
        s0 = min(per * self.rank, units)
        s1 = min(s0 + per, units)
        return s0 * 8, s1 * 8

    # ------------------------------------------------------------------ fused optimizer state
    def _init_fused_state(self):
        kind = self.fused
        for b in self.buckets:
            s0, s1 = self.shard_range(b)
            n = max(s1 - s0, 8)
            b.master = torch.zeros(n, dtype=torch.float32, device=self.device)
            b.master[: s1 - s0].copy_(b.flat_param[s0:s1].float())
            b.state0 = torch.zeros(n, dtype=torch.float32, device=self.device)
            b.state1 = torch.zeros(n, dtype=torch.float32, device=self.device) if kind != "sgd" else None
        ng = len(self.param_groups)
        # clip mode: one more row holds the ClipState {max_norm, norm, coef, step}, so refresh_hparams writes
        # max_norm together with the groups in one launch
        self._hp_dev = torch.zeros((ng + int(self.clip), 64), dtype=torch.uint8, device=self.device)
        self._group_step = [0] * ng
        self.loss_scale = 1.0
        if self.clip:
            self._init_clip()

    def _init_clip(self):
        cu = self.ctx.cu
        ng = len(self.param_groups)
        self._clip_state_ptr = self._hp_dev.data_ptr() + 64 * ng
        self._grad_norm = self._hp_dev[ng, 4:8].view(torch.float32)[0]
        # phase-1 partial sums, [bucket][CTA]; entries of CTAs a bucket does not launch stay zero
        self._clip_slots = torch.zeros(len(self.buckets) * cu.CLIP_SLOTS_PER_BUCKET, dtype=torch.float64,
                                       device=self.device)
        # phase 3: one static table of ClipDesc per dtype, built once (graph-safe)
        kind = cu.OPT_SGD if self.fused == "sgd" else cu.OPT_ADAM
        nstreams = 2 if kind == cu.OPT_SGD else 3
        by_dtype: Dict[torch.dtype, List[Bucket]] = {}
        for b in self.buckets:
            by_dtype.setdefault(b.dtype, []).append(b)
        self._clip_tables = []
        for dtype, bs in by_dtype.items():
            rows = [[b.grad_off, b.param_off, b.numel, b.master.data_ptr(), b.state0.data_ptr(),
                     b.state1.data_ptr() if b.state1 is not None else 0, self._hp_dev.data_ptr() + 64 * b.group_index,
                     0] for b in bs]
            table = torch.tensor(rows, dtype=torch.int64, device=self.device)
            assert table.element_size() * table.shape[1] == cu.CLIP_DESC_BYTES
            per_stage = nstreams * 256 * (16 // dtype.itemsize) * 4
            stages = max(2, min(8, (96 << 10) // per_stage))
            blocks = clip_update_grid([b.numel for b in bs], dtype.itemsize, self.world)
            self._clip_tables.append((wire_code(dtype), kind, table, len(bs), blocks, stages))

    def sync_master_from_params(self):
        for b in self.buckets:
            s0, s1 = self.shard_range(b)
            b.master[: s1 - s0].copy_(b.flat_param[s0:s1].float())

    def step_done(self):
        """Eager mode, end of optimizer.step(): count the step and publish the
        hyper-parameters of the next one."""
        if not self.fused or torch.cuda.is_current_stream_capturing():
            return
        for gi in range(len(self._group_step)):
            self._group_step[gi] += 1
        self.refresh_hparams()

    def pre_replay(self):
        """CUDA-graph mode, before every replay: publish the hyper-parameters of
        the step about to run, then count it."""
        if not self.fused:
            return
        self.refresh_hparams()
        for gi in range(len(self._group_step)):
            self._group_step[gi] += 1

    def refresh_hparams(self):
        """Send the param-group hyper-parameters (lr, momentum, Adam bias
        corrections, ...) of the NEXT step to the device block the fused kernels
        read.  The values ride in the argument space of a tiny kernel on the
        current stream, so they are ordered before the next exchange kernels and
        a captured CUDA graph sees fresh values on every replay."""
        if not self.fused:
            return
        cur = torch.cuda.current_stream(self.device)
        if torch.cuda.is_current_stream_capturing():
            return   # replays are fed from outside the graph
        blob = b""
        for gi, g in enumerate(self.param_groups):
            t = self._group_step[gi] + 1     # the step that is about to run
            if self.fused == "sgd":
                vals = (float(g.get("lr", 0.0)), float(g.get("weight_decay", 0.0)), float(g.get("momentum", 0.0)),
                        float(g.get("dampening", 0.0)), 0.0, 0.0, 0.0, 1.0, 1.0,
                        int(bool(g.get("nesterov", False))), 0, int(t == 1), 1.0 / self.loss_scale, 0, 0, 0)
            else:
                b1, b2 = g.get("betas", (0.9, 0.999))
                vals = (float(g.get("lr", 0.0)), float(g.get("weight_decay", 0.0)), 0.0, 0.0, float(b1), float(b2),
                        float(g.get("eps", 1e-8)), 1.0 - b1 ** t, 1.0 - b2 ** t, 0,
                        int(self.fused == "adamw"), int(t == 1), 1.0 / self.loss_scale, 0, 0, 0)
            blob += struct.pack(_HP_FMT, *vals)
        if self.clip:
            blob += struct.pack("<f", float(self.max_grad_norm))    # ClipState.max_norm, right behind the groups
        self.ctx.cu.write_blob(self._hp_dev.data_ptr(), blob, cur.cuda_stream)
        self.engine.launches += 1

    # ------------------------------------------------------------------ hooks
    def _register_hooks(self):
        for b in self.buckets:
            for p in b.params:
                self._hooks.append(p.register_post_accumulate_grad_hook(self._make_hook(p)))

    def _make_hook(self, p):
        def hook(param):
            if not self.enabled:
                return
            self._delay[p] -= 1
            if self._delay[p] > 0:
                return
            if self._delay[p] < 0:
                raise AssertionError(
                    "Gradients were computed more than backward_passes_per_step times before call to step(). "
                    "Increase backward_passes_per_step to accumulate gradients locally.")
            gv = self._grad_views[p]
            if p.grad is not gv:
                # someone replaced .grad (e.g. zero_grad(set_to_none=True)): fold it back into the arena
                if p.grad is not None and p.grad.data_ptr() != gv.data_ptr():
                    gv.copy_(p.grad)
                p.grad = gv
            b = self._param_bucket[p]
            b.pending -= 1
            if b.pending == 0:
                self._launch_ready(b)
        return hook

    def set_backward_passes_per_step(self, n: int):
        self.bpps = n
        for p in self._delay:
            self._delay[p] = n

    # ------------------------------------------------------------------ launching
    def _launch_ready(self, b: Optional[Bucket] = None):
        """Launch a bucket whose gradients are complete.  By default buckets go
        out in completion order - identical on every rank because autograd
        executes the same graph in the same order (the assumption DDP also
        makes); BYTEPS_STRICT_ORDER=1 forces creation order instead."""
        if b is not None and not self._strict:
            if not b.launched:
                self._issue(b)
            return
        while self._next < len(self.buckets) and self.buckets[self._next].pending == 0:
            if not self.buckets[self._next].launched:
                self._issue(self.buckets[self._next])
            self._next += 1

    def _issue(self, b: Bucket):
        if self._ring_mode == "off" or b.ring_cls is None:
            self._ring_flush()          # keep the comm stream in issue order
            self._launch(b)
        elif self._ring_mode == "persistent" and self._step >= self._ring_persistent_after:
            self._ring_persistent_ready(b)
        else:
            self._ring_enqueue(b)

    def _seg_table(self, b: Bucket) -> torch.Tensor:
        t = self._seg_tables.get(b.index)
        if t is None:
            ptr = b.flat_grad.data_ptr()
            t = torch.tensor([[ptr, ptr, 0, b.numel]], dtype=torch.int64, device=self.device)
            self._seg_tables[b.index] = t
        return t

    def _launch(self, b: Bucket):
        cu = self.ctx.cu
        view = self.ctx.view
        cur = torch.cuda.current_stream(self.device)
        tracing = (self.engine.timeline.enabled() and self.engine.timeline.active(self._step)
                   and not torch.cuda.is_current_stream_capturing())
        ev = torch.cuda.Event(enable_timing=tracing)
        ev.record(cur)
        cs = self.comm_stream
        cs.wait_event(ev)
        ev_t = None
        if tracing:
            ev_t = torch.cuda.Event(enable_timing=True)
            ev_t.record(cs)
        wire = self._wire(b)
        world = self.world
        scale = (1.0 / world) if self.average else 1.0
        wbytes = self._wire_bytes(b)
        shard = (wbytes + world - 1) // world
        blocks = self.engine.cfg.comm_blocks or pick_blocks(shard, self.threads, 32, cap=64)
        nvls = bool(self.ctx.nvls)
        if self.fused:
            kind = cu.OPT_SGD if self.fused == "sgd" else cu.OPT_ADAM
            hp_ptr = self._hp_dev.data_ptr() + 64 * b.group_index
            if self.clip:
                # phase 1 only: the update waits for the global norm (_clip_tail)
                slots = self._clip_slots.data_ptr() + 8 * cu.CLIP_SLOTS_PER_BUCKET * b.index
                cu.clip_reduce_sumsq(view, wire_code(wire), b.grad_off, b.numel, scale, slots, hp_ptr, blocks,
                                     self.threads, 0, nvls, cs.cuda_stream)
                self._after_launch(b, cur, cs, ev_t)
                return
            if wire == b.dtype and self._fused_engine == "tma":
                # optimizer state streamed through shared memory with bulk copies (pushpull.cu, TMA variant)
                es = 4 if b.dtype == torch.float32 else 2
                per_stage = (2 if kind == cu.OPT_SGD else 3) * 256 * (16 // es) * 4
                stages = max(2, min(8, (96 << 10) // per_stage))
                shard_units = (shard + 15) // 16
                cap = self._fused_tma_blocks
                tblocks = self.engine.cfg.comm_blocks or max(1, min(cap, (shard_units + 255) // 256))
                cu.pushpull_fused_opt_tma(view, wire_code(wire), kind, b.grad_off, b.param_off, b.numel, scale,
                                          b.master.data_ptr(), b.state0.data_ptr(),
                                          b.state1.data_ptr() if b.state1 is not None else 0, hp_ptr, tblocks, stages,
                                          nvls, 0, cs.cuda_stream)
                self._after_launch(b, cur, cs, ev_t)
                return
            if wire == b.dtype:
                segs, nsegs, stage = 0, 0, b.grad_off
            else:
                segs, nsegs, stage = self._seg_table(b).data_ptr(), 1, self.stage_off
            cu.pushpull_fused_opt(view, wire_code(b.dtype), wire_code(wire), wire_code(b.dtype), kind, segs, nsegs,
                                  stage, b.param_off, b.numel, scale, b.master.data_ptr(), b.state0.data_ptr(),
                                  b.state1.data_ptr() if b.state1 is not None else 0, hp_ptr, blocks, self.threads, 0,
                                  nvls, cs.cuda_stream)
        elif wire == b.dtype:
            eng_kind = self._reduce_engine
            if eng_kind == "tcgen05" and b.dtype in (torch.bfloat16, torch.float16) and world <= 8:
                # tensor-core reduction: TMA-fed [I|..|I] x [X_0;..;X_{P-1}] with a TMEM accumulator
                maps = self._umma_maps.get(b.index)
                if maps is None:
                    maps = cu.make_umma_maps(view, wire_code(wire), b.grad_off, b.numel)
                    self._umma_maps[b.index] = maps
                ublocks = max(1, min(64, (shard + 16383) // 16384))
                cu.pushpull_inplace_umma(view, maps, wire_code(wire), b.grad_off, b.numel, scale, ublocks, 0,
                                         cs.cuda_stream)
            elif eng_kind == "tma":
                tblocks = pick_blocks(shard, 256, 16, cap=64)
                cu.pushpull_inplace_tma(view, wire_code(wire), b.grad_off, b.numel, scale, tblocks, 4, 0,
                                        cs.cuda_stream)
            else:
                cu.pushpull_inplace(view, wire_code(wire), b.grad_off, b.numel, scale, blocks, self.threads, 0,
                                    nvls and eng_kind != "lsu", cs.cuda_stream)
        else:
            cu.pushpull_packed(view, wire_code(b.dtype), wire_code(wire), self._seg_table(b).data_ptr(), 1,
                               self.stage_off, b.numel, scale, blocks, self.threads, 0, nvls, False, True,
                               cs.cuda_stream)
        self._after_launch(b, cur, cs, ev_t)

    # ------------------------------------------------------------------ descriptor ring
    def _setup_ring(self):
        """BYTEPS_RING: how bucket exchanges reach the GPU.

        off         one kernel per bucket (two cross-rank barriers each);
        batch       buckets that became ready are handed to ONE descriptor-ring launch per flush window
                    (BYTEPS_RING_BATCH_BYTES, or the end of backward): flags instead of barriers, no
                    launch gaps, CTAs flow from one bucket into the next;
        persistent  one ring launch per step (per dtype class), issued when the first bucket is ready;
                    later buckets are announced by a `ring_mark` on the autograd stream.
        With BYTEPS_SCHEDULING_CREDIT > 0 the ring's root scheduler picks the ready bucket with the
        highest priority inside a byte-credit window (reference: scheduled_queue.cc:82-163)."""
        from ..ops.ring import RingEntry, RingTable

        cu = self.ctx.cu
        mode = os.environ.get("BYTEPS_RING", "auto").lower()
        if mode in ("0", "no", "false"):
            mode = "off"
        if mode in ("1", "yes", "true", "on"):
            mode = "batch"
        self._ring_tables = {}
        self._ring_pending: List[Bucket] = []
        self._ring_pending_bytes = 0
        self._ring_started = False
        self._ring_batch_bytes = _env_int("BYTEPS_RING_BATCH_BYTES", 64 << 20)
        # persistent launches spin while backward is still producing gradients.  CUDA loads kernels lazily and
        # a first-time load can wait for running kernels, so the first steps (which load cuDNN/cuBLAS/ATen
        # kernels) go through the batch path; the same step count on every rank keeps launches aligned.
        self._ring_persistent_after = _env_int("BYTEPS_RING_PERSISTENT_AFTER", 2)
        self._ring_blocks = _env_int("BYTEPS_RING_BLOCKS", 0)
        credit = self.engine.cfg.scheduling_credit
        self._ring_sched = credit > 0
        self._ring_credit = credit * self.engine.cfg.partition_bound() if credit > 0 else 0
        self._stamps = os.environ.get("BYTEPS_COMM_STAMPS", "1") not in ("0", "")
        self._stamp_base = None
        # clip mode has no ring variant: phase 1 goes out per bucket
        eligible = (not self.clip and self._reduce_engine in ("auto", "nvls", "lsu")
                    and len(self.buckets) <= cu.RING_SLOTS
                    and not (self.fused and self._fused_engine == "tma" and self.world == 1 and mode == "auto"))
        if mode == "auto":
            # one rank: nothing to wait for, the TMA-streamed optimizer kernel per bucket is the fastest;
            # several ranks: the ring removes two NVLink barrier round trips and a launch per bucket
            mode = "batch" if (self.world > 1 and eligible) else "off"
        if mode != "off" and not eligible:
            mode = "off"
        self._ring_mode = mode
        if mode == "off":
            return
        kind = {None: cu.RING_ALLREDUCE, "sgd": cu.RING_SGD}.get(self.fused, cu.RING_ADAM)
        scale = (1.0 / self.world) if self.average else 1.0
        by_cls = {}
        for b in self.buckets:
            if self._wire(b) != b.dtype:
                continue            # needs a wire cast: stays on the per-bucket packed kernel
            cls = (wire_code(b.dtype), kind)
            by_cls.setdefault(cls, []).append(b)
        for cls, bs in by_cls.items():
            entries = []
            for pos, b in enumerate(bs):
                b.ring_cls, b.ring_pos = cls, pos
                entries.append(RingEntry(
                    grad_off=b.grad_off, param_off=max(b.param_off, 0), numel=b.numel, wire=cls[0], slot=b.index,
                    kind=kind, scale=scale, priority=b.priority,
                    master=b.master.data_ptr() if b.master is not None else 0,
                    state0=b.state0.data_ptr() if b.state0 is not None else 0,
                    state1=b.state1.data_ptr() if b.state1 is not None else 0,
                    hp=(self._hp_dev.data_ptr() + 64 * b.group_index) if self.fused else 0))
            self._ring_tables[cls] = (RingTable(entries, self.device), bs)

    def _ring_grid(self, nbytes: int) -> int:
        if self._ring_blocks:
            return self._ring_blocks
        if self.engine.cfg.comm_blocks:
            return self.engine.cfg.comm_blocks
        shard = (nbytes + self.world - 1) // self.world
        return pick_blocks(shard, 512, 32, cap=64 if self._ring_mode == "batch" else 24)

    def _ring_enqueue(self, b: Bucket):
        """batch mode: remember the bucket; flush when enough bytes are waiting."""
        self._ring_pending.append(b)
        self._ring_pending_bytes += b.nbytes
        b.launched = True
        self._launched += 1
        if self._ring_pending_bytes >= self._ring_batch_bytes:
            self._ring_flush()
        elif self.auto_finish is not None and self._launched == len(self.buckets):
            self._ring_flush()
            self.auto_finish()

    def _ring_flush(self):
        """One ring launch per run of pending buckets that are consecutive in their class table."""
        pend = self._ring_pending
        if not pend:
            return
        self._ring_pending = []
        self._ring_pending_bytes = 0
        cur = torch.cuda.current_stream(self.device)
        cs = self.comm_stream
        ev = torch.cuda.Event()
        ev.record(cur)
        cs.wait_event(ev)
        nvls = bool(self.ctx.nvls) and self._reduce_engine != "lsu"
        i = 0
        while i < len(pend):
            b0 = pend[i]
            j = i + 1
            while (j < len(pend) and pend[j].ring_cls == b0.ring_cls
                   and pend[j].ring_pos == pend[j - 1].ring_pos + 1):
                j += 1
            table, _ = self._ring_tables[b0.ring_cls]
            nbytes = sum(x.nbytes for x in pend[i:j])
            table.launch(self.ctx.view, self._ring_grid(nbytes // max(1, j - i)), cs.cuda_stream, nvls=nvls,
                         sched=self._ring_sched and j - i > 1, self_mark=True, credit_bytes=self._ring_credit,
                         first=b0.ring_pos, count=j - i)
            self._count_launch()
            i = j
        done = torch.cuda.Event()
        done.record(cs)
        for b in pend:
            b.done = done
            if self.engine.telemetry.should_record():
                self.engine.telemetry.record(b.nbytes)
        self._last_done = done
        self._ring_traced = True

    def _ring_persistent_ready(self, b: Bucket):
        """persistent mode: the first ready bucket of a step starts one ring launch per class (they
        consume their tables in order and wait on flags); every ready bucket is announced by a mark
        kernel on the producing stream."""
        cur = torch.cuda.current_stream(self.device)
        cs = self.comm_stream
        self.ctx.cu.ring_mark(self.ctx.view, [b.index], cur.cuda_stream)
        self._count_launch()
        if not self._ring_started:
            self._ring_started = True
            ev = torch.cuda.Event()
            ev.record(cur)
            cs.wait_event(ev)
            nvls = bool(self.ctx.nvls) and self._reduce_engine != "lsu"
            for cls, (table, bs) in self._ring_tables.items():
                nbytes = sum(x.nbytes for x in bs) // len(bs)
                table.launch(self.ctx.view, self._ring_grid(nbytes), cs.cuda_stream, nvls=nvls,
                             sched=self._ring_sched and len(bs) > 1, self_mark=False,
                             credit_bytes=self._ring_credit)
                self._count_launch()
            done = torch.cuda.Event()
            done.record(cs)
            self._last_done = done
            for x in self.buckets:
                if x.ring_cls is not None:
                    x.done = done
        if self.engine.telemetry.should_record():
            self.engine.telemetry.record(b.nbytes)
        b.launched = True
        self._launched += 1
        self._ring_traced = True
        if self.auto_finish is not None and self._launched == len(self.buckets):
            self.auto_finish()

    def exposed_comm_ms(self) -> Optional[float]:
        """Device-measured communication time that was NOT hidden behind the backward pass in the
        last step: (comm stream idle after the last exchange) - (autograd stream reached
        optimizer.step), both stamped with the GPU's globaltimer by one-thread kernels, so the
        figure also exists for CUDA-graph replays.  None before the first step."""
        if not self._stamps:
            return None
        torch.cuda.synchronize(self.device)
        _, stamps = self.ctx.cu.ring_trace(self.ctx.view, [])
        if stamps[0] == 0 or stamps[1] == 0:
            return None
        return max(0.0, (stamps[1] - stamps[0]) / 1e6)

    def ring_spans(self):
        """[(bucket index, order position, start ns, end ns)] of the last ring launches (globaltimer)."""
        torch.cuda.synchronize(self.device)
        idx = [b.index for b in self.buckets if b.ring_cls is not None]
        rows, _ = self.ctx.cu.ring_trace(self.ctx.view, idx)
        return [(i, pos, t0, t1) for i, (pos, t0, t1) in zip(idx, rows)]

    def _count_launch(self, n: int = 1):
        self.engine.launches += n
        self._xlaunches += n

    def launches_per_step(self) -> int:
        """Kernels of ours (exchange launches + marks) the last completed step issued; what one
        CUDA-graph replay of that step launches."""
        return self._last_step_launches

    def _after_launch(self, b: Bucket, cur, cs, ev_t):
        self._count_launch()
        if self.engine.telemetry.should_record():
            self.engine.telemetry.record(b.nbytes)
        tl = self.engine.timeline
        if tl.enabled() and tl.active(self._step) and not torch.cuda.is_current_stream_capturing():
            # device-timed span of this bucket's exchange (the reference's timeline uses host wall-clock)
            if self._trace_t0 is None:
                self._trace_t0 = (torch.cuda.Event(enable_timing=True), self.engine.core.now_us())
                self._trace_t0[0].record(cur)
            b.done = torch.cuda.Event(enable_timing=True)
            b.done.record(cs)
            self._trace_spans.append((b, ev_t, b.done))
        else:
            b.done = torch.cuda.Event()
            b.done.record(cs)
        b.launched = True
        self._last_done = b.done
        self._launched += 1
        if self.auto_finish is not None and self._launched == len(self.buckets):
            self.auto_finish()

    def synchronize(self):
        """Issue whatever has not been launched (unused parameters) and make the
        current stream wait for every bucket of this step."""
        cur = torch.cuda.current_stream(self.device)
        if self._stamps:
            self.ctx.cu.ring_stamp(self.ctx.view, 0, cur.cuda_stream)       # backward (and everything before) done
            self._count_launch()
        for b in self.buckets:
            if not b.launched:      # unused parameters: issue in index order on every rank
                self._zero_unused(b)
                b.pending = 0
                self._issue(b)
        self._ring_flush()
        self._clip_tail()
        if self._stamps and self._last_done is not None:
            self.ctx.cu.ring_stamp(self.ctx.view, 1, self.comm_stream.cuda_stream)   # last exchange finished
            self._count_launch()
            self._last_done = torch.cuda.Event()
            self._last_done.record(self.comm_stream)
        if self._last_done is not None:
            # the comm stream executes in order: the most recent event covers every bucket
            torch.cuda.current_stream(self.device).wait_event(self._last_done)
            self._last_done = None
        self._reset()

    def _zero_unused(self, b: Bucket):
        """A parameter whose hook did not fire in this iteration contributes zeros (like a fresh zero gradient in the
        reference), not whatever an earlier iteration left in its arena window - `model.zero_grad()` only drops the
        `.grad` references, it does not clear the arena."""
        for p in b.params:
            if self._delay.get(p) == self.bpps:
                self._grad_views[p].zero_()

    def finish_launches(self):
        """Launch every bucket that has not gone out yet, without waiting."""
        for b in self.buckets:
            if not b.launched:
                self._zero_unused(b)
                b.pending = 0
                self._issue(b)
        self._ring_flush()
        self._clip_tail()
        if self._stamps and self._last_done is not None:
            self.ctx.cu.ring_stamp(self.ctx.view, 1, self.comm_stream.cuda_stream)   # last exchange finished
            self._count_launch()
        self._reset(keep_events=True)

    def _clip_tail(self):
        """Clip mode, after every bucket's phase 1: the global norm (phase 2), then the clipped update and parameter
        all-gather (phase 3) on the comm stream.  The comm stream first waits for the current stream, so the new
        parameters cannot land under a kernel of this step that still reads the old ones."""
        if not self.clip:
            return
        cu, view, cs = self.ctx.cu, self.ctx.view, self.comm_stream
        cs.wait_stream(torch.cuda.current_stream(self.device))
        cu.clip_finalize(view, self._clip_slots.data_ptr(), self._clip_slots.numel(), self.clip_pub_off,
                         self._clip_state_ptr, 0, cs.cuda_stream)
        nvls = bool(self.ctx.nvls)
        for wire, kind, table, n, blocks, stages in self._clip_tables:
            cu.clip_update(view, wire, kind, table.data_ptr(), n, self._clip_state_ptr, blocks, stages, nvls, 0,
                           cs.cuda_stream)
        self._count_launch(1 + len(self._clip_tables))
        done = torch.cuda.Event()
        done.record(cs)
        for b in self.buckets:        # the parameters of every bucket change only now
            b.done = done
        self._last_done = done

    def grad_norm(self) -> torch.Tensor:
        """Clip mode: 0-dim fp32 device tensor with the total gradient norm of the last step (before clipping).
        Always the same storage, so CUDA-graph replays update it."""
        return self._grad_norm

    def _flush_trace(self):
        """Turn the timing events of this step into Chrome-trace spans (device time, anchored at
        the host timestamp of the step's first launch)."""
        if not self._trace_spans:
            return
        tl = self.engine.timeline
        t0_ev, t0_us = self._trace_t0
        self._trace_spans[-1][2].synchronize()
        for b, start, end in self._trace_spans:
            ts = t0_us + int(t0_ev.elapsed_time(start) * 1000)
            dur = max(1, int(start.elapsed_time(end) * 1000))
            name = "bucket%d[%s x%d]" % (b.index, str(b.dtype)[6:], len(b.params))
            stage = "PUSHPULL_FUSED_OPT" if self.fused else "PUSHPULL"
            tl.record(name, stage, b.index, ts, dur)
            tl.record(name, "", (1 << 64) - 1, ts, dur)
        self._trace_spans = []
        self._trace_t0 = None
        if self._step + 1 >= tl.end_step():
            tl.dump()

    def record_ring_trace(self, dump: bool = False):
        """Chrome-trace spans of the last step's ring launches.  The kernels stamp the GPU's
        globaltimer when the first CTA picks a bucket up and when the last CTA finishes it, so the
        spans exist for CUDA-graph replays too (the reference's timeline is host wall-clock only,
        docs/timeline.md; events cannot be recorded inside a captured graph)."""
        tl = self.engine.timeline
        if not tl.enabled() or not getattr(self, "_ring_traced", False):
            return
        if self._stamp_base is None:
            # anchor: one stamp kernel + the host clock right after it completed
            self.ctx.cu.ring_stamp(self.ctx.view, 15, torch.cuda.current_stream(self.device).cuda_stream)
            torch.cuda.synchronize(self.device)
            host_us = self.engine.core.now_us()
            _, st = self.ctx.cu.ring_trace(self.ctx.view, [])
            self._stamp_base = (host_us, st[15])
        host_us, gt0 = self._stamp_base
        by_index = {b.index: b for b in self.buckets}
        for idx, pos, t0, t1 in self.ring_spans():
            if t1 <= t0 or t0 == 0:
                continue
            b = by_index[idx]
            ts = host_us + (int(t0) - int(gt0)) // 1000
            dur = max(1, (int(t1) - int(t0)) // 1000)
            name = "bucket%d[%s x%d prio %d #%d]" % (b.index, str(b.dtype)[6:], len(b.params), b.priority, pos)
            tl.record(name, "PUSHPULL_FUSED_OPT" if self.fused else "PUSHPULL", b.index, ts, dur)
            tl.record(name, "", (1 << 64) - 1, ts, dur)
        self._ring_traced = False
        if dump or self._step + 1 >= tl.end_step():
            tl.dump()

    def _reset(self, keep_events: bool = False):
        self._flush_trace()
        if (self._ring_mode != "off" and self.engine.timeline.enabled() and self.engine.timeline.active(self._step)
                and not torch.cuda.is_current_stream_capturing()):
            self.record_ring_trace()
        self._launched = 0
        self._next = 0
        self._step += 1
        self._ring_started = False
        self._last_step_launches, self._xlaunches = self._xlaunches, 0
        for b in self.buckets:
            b.pending = len(b.params)
            b.launched = False
        for p in self._delay:
            self._delay[p] = self.bpps

    def zero_grad(self):
        for b in self.buckets:
            b.flat_grad.zero_()

    def remove_hooks(self):
        for h in self._hooks:
            h.remove()
        self._hooks = []

    # ------------------------------------------------------------------ state access (fused mode)
    def master_params(self) -> Dict[torch.nn.Parameter, torch.Tensor]:
        """fp32 master values of THIS rank's shard, keyed by parameter (partial views)."""
        out = {}
        for b in self.buckets:
            s0, s1 = self.shard_range(b)
            for p, st in zip(b.params, b.starts):
                lo, hi = max(st, s0), min(st + p.numel(), s1)
                if lo < hi:
                    out[p] = (lo - st, b.master[lo - s0:hi - s0])
        return out

    def close(self):
        self.remove_hooks()
        torch.cuda.synchronize(self.device)
        for b in self.buckets:
            for p in b.params:
                if p.grad is not None:
                    p.grad = p.grad.detach().clone()
                if self.fused:
                    p.data = p.data.clone()
        if self.world > 1:
            self.engine.group.barrier()
        self.ctx.close()
