#!/usr/bin/env python
"""Headline benchmark: data-parallel ResNet-50 (bf16) synthetic training throughput.

This is the reference's own benchmark (/root/reference/example/pytorch/benchmark_byteps.py:
torchvision-style ResNet-50, synthetic 3x224x224 batches, SGD lr=0.01 wrapped in
``DistributedOptimizer``, img/sec = batch * steps / time, total = per-GPU * size),
run through OUR public API, in the configuration BASELINE.json names
("ResNet-50 data-parallel bf16 on 8xB200"; batch 64 per GPU as in the
reference's published ResNet-50 numbers, docs/performance.md).

    python bench.py --gpus 1 --steps 50 --warmup 10
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 50 --warmup 10

Prints ONE JSON line on rank 0.  `value` is the whole-job images/s measured on
the device (CUDA events, max over ranks); `e2e` is the same loop including the
per-step H2D copy of the inputs from pinned host memory and a D2H read of the
loss.  `--impl reference` reports that the unmodified reference cannot be
installed offline (see DESIGN.md); `--impl nccl` runs the reference-STYLE NCCL
path (per-partition reduce-scatter/all-gather + div, unfused optimizer) and
`--impl ddp` the strongest library baseline on the same box (torch DDP, NCCL
bucketed all-reduce, fused torch optimizer, whole step captured in the same
CUDA graph) for our own comparison tables.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "nccl", "ddp"],
                    help="ours: byteps_b200; reference: the unmodified bytedance/byteps (not installable offline); "
                         "nccl: reference-STYLE per-partition NCCL path; ddp: torch DDP + NCCL bucketed all-reduce + "
                         "fused torch optimizer, whole step in the same CUDA graph (the fair same-box baseline)")
    ap.add_argument("--model", default="resnet50")
    ap.add_argument("--batch-size", type=int, default=64, help="per-GPU batch (weak scaling)")
    ap.add_argument("--seq-len", type=int, default=128, help="BERT models only")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-graph", action="store_true", help="disable whole-step CUDA graph capture")
    ap.add_argument("--no-fused", action="store_true", help="unfused optimizer (gradient all-gather + torch step)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cudnn-benchmark", action="store_true",
                    help="cuDNN autotuning: measured no faster than the heuristics on B200 (14.2 vs 14.1 ms/step) "
                         "and 25-45 s slower to start")
    ap.add_argument("--verbose", action="store_true", help="phase progress on stderr (all ranks)")
    ap.add_argument("--hang-dump", type=float, default=float(os.environ.get("BENCH_HANG_DUMP_S", "0")),
                    help="dump python stacks of every thread to stderr every N seconds (debugging hangs)")
    ap.add_argument("--momentum", type=float, default=0.0)
    ap.add_argument("--optimizer", default="auto", choices=["auto", "sgd", "adamw"],
                    help="auto: SGD lr=0.01 for CNNs (the reference benchmark), AdamW for BERT")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the device-timed steps, write what the last of them computed on rank 0 to "
                         "DIR/<name>.npy (float32): its loss and a fixed sample of the updated parameters")
    return ap.parse_args()


def dump_outputs(out_dir, torch, loss, model, max_params=1 << 22):
    """loss.npy: the step's loss.  params.npy: the parameters after the step's update, flattened and concatenated in
    model.parameters() order; above ``max_params`` values, the values at a fixed, seeded set of positions (sorted),
    which keeps the files under 64 MB for any model."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().reshape(1).cpu().numpy())
    flat = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()])
    if flat.numel() > max_params:
        idx = torch.randint(0, flat.numel(), (max_params,), generator=torch.Generator().manual_seed(0)).unique()
        flat = flat[idx.to(flat.device)]
    np.save(os.path.join(out_dir, "params.npy"), flat.cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:  # noqa: BLE001
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.strip().split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except ValueError:
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class _TorchDist:
    """rank()/size()/init()/shutdown() of the DDP arm: plain torch.distributed, none of our engine."""

    def __init__(self, torch, world, local_rank):
        self.torch, self.world, self.local_rank = torch, world, local_rank

    def init(self):
        if self.world > 1:
            import torch.distributed as dist

            os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")   # required for NCCL under graph capture
            dist.init_process_group("nccl", device_id=self.torch.device("cuda", self.local_rank))

    def rank(self):
        return int(os.environ.get("RANK", "0"))

    def size(self):
        return self.world

    def shutdown(self):
        # destroy_process_group() blocks forever while captured NCCL graphs are alive (observed on 2 GPUs): the
        # arm has printed its line, so synchronise and leave without tearing NCCL down
        if self.world > 1:
            import torch.distributed as dist

            self.torch.cuda.synchronize()
            dist.barrier()
            self.torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def build(args, torch, bps, device):
    from byteps_b200.models import get_model

    is_bert = args.model.startswith("bert")
    torch.manual_seed(1234)     # same initial weights on every run, so that two builds compute the same steps
    model = get_model(args.model)
    dt = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    model = model.to(device)
    if not is_bert:
        model = model.to(memory_format=torch.channels_last)
    if dt != torch.float32:
        model = model.to(dt)
        for m in model.modules():   # keep normalisation statistics/affine in fp32 (cuDNN mixed-dtype path)
            if isinstance(m, (torch.nn.BatchNorm2d,)):
                m.float()
    model.train()
    B = args.batch_size
    gen = torch.Generator().manual_seed(1234 + bps.rank())
    nbuf = 4
    if is_bert:
        S = args.seq_len
        host = [(torch.randint(0, 30522, (B, S), generator=gen).pin_memory(),
                 torch.randint(0, 30522, (B, S), generator=gen).pin_memory()) for _ in range(nbuf)]
    else:
        host = [(torch.rand(B, 3, 224, 224, generator=gen).to(dt).contiguous(memory_format=torch.channels_last)
                 .pin_memory(), torch.randint(0, 1000, (B,), generator=gen).pin_memory()) for _ in range(nbuf)]
    static_x = host[0][0].to(device, non_blocking=True)
    static_y = host[0][1].to(device, non_blocking=True)
    return model, host, static_x, static_y, is_bert


def main():
    args = parse()
    if args.impl == "reference":
        if os.environ.get("RANK", "0") != "0":      # under torchrun only rank 0 reports
            return 0
        print(json.dumps({"impl": "reference",
                          "unavailable": "bytedance/byteps cannot be installed offline: its ps-lite build downloads "
                                         "ZeroMQ and its torch plugin needs TH/THC headers removed from torch>=2 "
                                         "(see DESIGN.md)"}))
        return 0
    if args.hang_dump > 0:
        import faulthandler

        faulthandler.dump_traceback_later(args.hang_dump, repeat=True, file=sys.stderr)
    t_start = time.time()

    def note(what):
        if args.verbose:
            sys.stderr.write("[bench r%s +%.1fs] %s\n" % (os.environ.get("RANK", "0"), time.time() - t_start, what))
            sys.stderr.flush()

    import torch
    import torch.nn.functional as F

    import byteps_b200.torch as bps
    from byteps_b200.torch.graph import GraphedStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            # convenience: re-launch under torchrun
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
                   "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
            return subprocess.call(cmd)
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    torch.backends.cudnn.benchmark = bool(args.cudnn_benchmark)
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    if args.impl == "nccl":
        os.environ["BYTEPS_BACKEND"] = "nccl"
    note("torch imported")
    is_ddp = args.impl == "ddp"
    if is_ddp:
        bps = _TorchDist(torch, world, local_rank)      # noqa: F811 - the baseline arm must not touch our engine
    bps.init()
    note("init done")
    model, host, sx, sy, is_bert = build(args, torch, bps, device)
    note("model built")
    fused = not args.no_fused and args.impl == "ours"
    opt_name = args.optimizer if args.optimizer != "auto" else ("adamw" if is_bert else "sgd")
    fwd_model = model
    if is_ddp:
        # library baseline: bucketed NCCL all-reduce overlapped with backward by DDP's reducer, torch's fused
        # (single multi-tensor kernel) optimizers, same whole-step CUDA graph as our arm
        if opt_name == "adamw":
            opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.01, fused=True, capturable=True)
        else:
            opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=args.momentum, fused=True)
        if world > 1:
            side = torch.cuda.Stream(device=device)
            side.wait_stream(torch.cuda.current_stream(device))
            with torch.cuda.stream(side):               # DDP must be built on a side stream to be graph-capturable
                fwd_model = torch.nn.parallel.DistributedDataParallel(
                    model, device_ids=[local_rank], gradient_as_bucket_view=True, static_graph=True,
                    broadcast_buffers=False)
            torch.cuda.current_stream(device).wait_stream(side)
    else:
        if opt_name == "adamw":
            base = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.01)
        else:
            base = torch.optim.SGD(model.parameters(), lr=0.01, momentum=args.momentum)
        opt = bps.DistributedOptimizer(base, named_parameters=model.named_parameters(), fused_update=fused)
        note("optimizer wrapped")
        bps.broadcast_parameters(model.state_dict(), root_rank=0)
        note("parameters broadcast")
        if not fused:
            bps.broadcast_optimizer_state(opt, root_rank=0)

    def train_step():
        opt.zero_grad(set_to_none=False) if is_ddp else opt.zero_grad()
        if is_bert:
            loss = fwd_model(sx, mlm_labels=sy)
        else:
            loss = F.cross_entropy(fwd_model(sx).float(), sy)
        loss.backward()
        opt.step()
        return loss

    eng = None if is_ddp else __import__("byteps_b200.common", fromlist=["engine"]).engine()
    use_graph = not args.no_graph and args.impl in ("ours", "ddp")
    graph_note = None
    if use_graph and is_ddp:
        try:
            # DDP needs >= 11 eager iterations before capture (torch CUDA-graphs notes)
            stepper = GraphedStep(train_step, warmup=11, device=device)
        except Exception as e:  # noqa: BLE001 - report the arm eager rather than not at all
            graph_note = "capture failed (%s); eager" % str(e).splitlines()[0][:120]
            use_graph = False
            torch.cuda.synchronize(device)
            stepper = train_step
    elif use_graph:
        stepper = GraphedStep(train_step, warmup=3, pre_replay=opt.refresh_hparams if fused else None, device=device)
    else:
        stepper = train_step

    def sync_all():
        torch.cuda.synchronize(device)
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
            torch.cuda.synchronize(device)

    def timed(loop_body, steps):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            loop_body(i)
        e1.record()
        torch.cuda.synchronize(device)
        ms = e0.elapsed_time(e1)
        if world > 1:
            import torch.distributed as dist

            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        sync_all()
        return ms

    note("graph captured" if use_graph else "eager stepper")
    # ---- warm-up (untimed)
    for i in range(max(args.warmup, 3)):
        stepper()
    torch.cuda.synchronize(device)
    note("warm-up done")
    launches0 = eng.launches if eng is not None else 0
    replay_launches = None
    sampler = ClockSampler(local_rank)
    if bps.rank() == 0:
        sampler.start()
    # ---- device-timed region: inputs resident on the device (the reference's benchmark does the same)
    last_loss = [None]

    def timed_step(i):
        last_loss[0] = stepper()
    ms = timed(timed_step, args.steps)
    note("device-timed region done: %.3f ms/step" % (ms / args.steps))
    if args.dump_outputs and bps.rank() == 0:
        dump_outputs(args.dump_outputs, torch, last_loss[0], model)
        note("outputs written to %s" % args.dump_outputs)
    if use_graph:
        # kernels of ours inside one captured step (graph replays do not pass through python launch counters)
        gs = getattr(opt, "grad_sync", None)
        # kernels of ours inside one replay = what one eager step launched (counted during GraphedStep's warm-up)
        replay_launches = (gs.launches_per_step() + (1 if fused else 0)) * args.steps if gs is not None else 0
    gpu_launches = replay_launches if use_graph else (eng.launches - launches0 if eng is not None else 0)
    if args.impl in ("nccl", "ddp"):
        gpu_launches = 0     # the comparison arms run NCCL's kernels, none of ours
    # communication NOT hidden behind backward, stamped on the device (works under graph replay)
    exposed = None
    if args.impl == "ours" and getattr(opt, "grad_sync", None) is not None:
        exposed = opt.grad_sync.exposed_comm_ms()
    # ---- end-to-end region: per-step H2D of the batch from pinned memory + D2H read of the loss
    e2e = None
    if not args.no_e2e:
        # Every step: H2D copy of that step's batch from pinned host memory + D2H read of its loss.
        # Both are pipelined like a real input pipeline would: batch i+1 is prefetched on a copy
        # stream while step i computes, and the loss of step i is read (blocking) right after step
        # i+1 has been enqueued, so the GPU never idles on the host.
        copy_stream = torch.cuda.Stream(device=device)
        stage_x, stage_y = torch.empty_like(sx), torch.empty_like(sy)
        loss_host = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = torch.cuda.Event()
        losses = []
        state = {"pending": None}

        def prefetch(i):
            x, y = host[i % len(host)]
            copy_stream.wait_event(consumed)          # previous batch has left the staging buffers
            with torch.cuda.stream(copy_stream):
                stage_x.copy_(x, non_blocking=True)
                stage_y.copy_(y, non_blocking=True)

        def body(i):
            cur = torch.cuda.current_stream(device)
            cur.wait_stream(copy_stream)
            sx.copy_(stage_x, non_blocking=True)
            sy.copy_(stage_y, non_blocking=True)
            consumed.record(cur)
            prefetch(i + 1)
            loss = stepper()
            slot = i & 1
            loss_host[slot].copy_(loss.detach().float().reshape(1), non_blocking=True)   # D2H of this step's loss
            loss_ev[slot].record(cur)
            if state["pending"] is not None:          # blocking host read of the PREVIOUS step's loss
                ps = state["pending"]
                loss_ev[ps].synchronize()
                losses.append(float(loss_host[ps][0]))
            state["pending"] = slot

        def drain():
            if state["pending"] is not None:
                loss_ev[state["pending"]].synchronize()
                losses.append(float(loss_host[state["pending"]][0]))
                state["pending"] = None

        consumed.record(torch.cuda.current_stream(device))
        prefetch(0)
        for i in range(3):
            body(i)
        drain()

        def e2e_loop(i):
            body(i)
            if i == args.steps - 1:
                drain()                               # the last loss is read inside the timed region too
        ms_e2e = timed(e2e_loop, args.steps)
        note("e2e region done: %.3f ms/step" % (ms_e2e / args.steps))
        h2d = host[0][0].numel() * host[0][0].element_size() + host[0][1].numel() * host[0][1].element_size()
        unit_n = args.batch_size * (args.seq_len if is_bert else 1)
        e2e = {"value": unit_n * world * args.steps / (ms_e2e / 1e3), "unit": "tokens/s" if is_bert else "img/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps,
               "pipeline": "H2D of batch i+1 prefetched on a copy stream during step i; loss of step i read "
                           "(blocking) after step i+1 is enqueued; %d losses read" % len(losses),
               "last_loss": losses[-1] if losses else None}
    clocks = sampler.stop() if bps.rank() == 0 else None
    unit_n = args.batch_size * (args.seq_len if is_bert else 1)
    value = unit_n * world * args.steps / (ms / 1e3)
    if bps.rank() == 0:
        nparams = sum(p.numel() for p in model.parameters())
        out = {
            "metric": ("%s data-parallel training throughput (synthetic %s, %s, DistributedOptimizer)"
                       % (args.model, "tokens" if is_bert else "images", "AdamW" if opt_name == "adamw" else "SGD")),
            "value": value, "unit": "tokens/s" if is_bert else "img/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "impl": args.impl,
            "config": {"model": args.model, "global_batch": args.batch_size * world,
                       "per_gpu_batch": args.batch_size, "seq_len": args.seq_len if is_bert else None,
                       "parallelism": "dp%d" % world,
                       "optimizer": ("AdamW lr=1e-4 wd=0.01" if opt_name == "adamw"
                                     else "SGD lr=0.01 momentum=%g" % args.momentum),
                       "fused_update": fused, "cuda_graph": use_graph, "params": nparams,
                       "l2": "no explicit flush: a step streams weights+activations+gradients far larger than "
                             "the 126 MB L2",
                       "backend": eng.backend if eng is not None else "torch DDP + NCCL",
                       "ring": getattr(getattr(opt, "grad_sync", None), "_ring_mode", None),
                       "graph_note": graph_note},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(gpu_launches), "exposed_comm_ms": exposed,
        }
        print(json.dumps(out))
        sys.stdout.flush()
    bps.shutdown()
    note("shutdown done")
    return 0


if __name__ == "__main__":
    sys.exit(main())
