"""What global-norm gradient clipping costs on the fused path.

BERT-large, bf16 weights, AdamW, at bench.py's shapes (per-GPU batch 64, sequence 128); the whole step (zero_grad,
forward, backward, optimizer) is captured in one CUDA graph and device-timed.  One call alternates the arms round by
round, so they share the machine's state:

  fused         DistributedOptimizer(fused_update=True): update inside the exchange kernels, no clipping
  fused_clip    the same with max_grad_norm: norm on the device between the reduction and the update
  unfused_clip  fused_update=False with the same max_grad_norm: clip_grad_norm_ + torch's AdamW (capturable)
  ddp_clip      (world > 1) torch DDP + NCCL + torch's fused AdamW + clip_grad_norm_ in the same graph

Per arm: ms/step (max over ranks, median over rounds) and exposed_comm_ms (our arms).  fused_clip and unfused_clip
also run the same seeded steps from the same weights, and their parameters are compared within a bf16 tolerance.
The GPU name and power limit are read in the same run.

    python benchmarks/clip_bench.py --gpus 1
    python benchmarks/clip_bench.py --gpus 8      # re-launches itself under torchrun
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed graph replays per arm and round")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch-size", type=int, default=64)
    ap.add_argument("--seq-len", type=int, default=128)
    ap.add_argument("--max-grad-norm", type=float, default=1.0)
    ap.add_argument("--check-steps", type=int, default=1,
                    help="seeded steps of the fused_clip vs unfused_clip check.  One step compares like with like: "
                         "afterwards the trajectories part, because the fused path keeps fp32 master weights and "
                         "torch's AdamW updates the bf16 weights in place")
    return ap.parse_args()


def gpu_info(torch, device):
    name = torch.cuda.get_device_name(device)
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(device.index), "--query-gpu=power.limit",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        power = float(out.strip().splitlines()[0])
    except Exception:  # noqa: BLE001 - reported as unknown rather than guessed
        power = None
    return name, power


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
                   "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
            return subprocess.call(cmd)
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    import torch

    import byteps_b200.torch as bps
    from byteps_b200.models import get_model
    from byteps_b200.torch.graph import GraphedStep

    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    torch.backends.cuda.matmul.allow_tf32 = True
    bps.init()
    rank = bps.rank()
    B, S, mn = args.batch_size, args.seq_len, args.max_grad_norm

    def make_model():
        torch.manual_seed(1234)
        return get_model("bert_large").to(device).to(torch.bfloat16).train()

    gen = torch.Generator(device=device).manual_seed(1234 + rank)
    sx = torch.randint(0, 30522, (B, S), device=device, generator=gen)
    sy = torch.randint(0, 30522, (B, S), device=device, generator=gen)

    arms = {}

    def add_ours(name, fused, clip):
        model = make_model()
        base = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.01, capturable=not fused)
        opt = bps.DistributedOptimizer(base, named_parameters=model.named_parameters(), fused_update=fused,
                                       max_grad_norm=mn if clip else None)
        bps.broadcast_parameters(model.state_dict(), root_rank=0)
        arms[name] = {"model": model, "opt": opt, "fwd": model, "fused": fused}

    add_ours("fused", True, False)
    add_ours("fused_clip", True, True)
    add_ours("unfused_clip", False, True)
    if world > 1:
        model = make_model()
        opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.01, fused=True, capturable=True)
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):     # DDP must be built on a side stream to be graph-capturable
            ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank],
                                                            gradient_as_bucket_view=True, static_graph=True,
                                                            broadcast_buffers=False)
        torch.cuda.current_stream(device).wait_stream(side)
        arms["ddp_clip"] = {"model": model, "opt": opt, "fwd": ddp, "fused": None}

    def step_fn(arm):
        model, opt, fwd = arm["model"], arm["opt"], arm["fwd"]

        def step():
            opt.zero_grad(set_to_none=False) if arm["fused"] is None else opt.zero_grad()
            loss = fwd(sx, mlm_labels=sy)
            loss.backward()
            if arm["fused"] is None:
                torch.nn.utils.clip_grad_norm_(model.parameters(), mn)
            opt.step()
            return loss
        return step

    def sync_all():
        torch.cuda.synchronize(device)
        if world > 1:
            torch.distributed.barrier()
            torch.cuda.synchronize(device)

    # ---- correctness: fused_clip vs unfused_clip on the same seeded steps, eager, from the same weights
    check = {}
    for name in ("fused_clip", "unfused_clip"):
        st = step_fn(arms[name])
        torch.manual_seed(4321)      # the same dropout masks in both arms
        for _ in range(args.check_steps):
            st()
        sync_all()
        check[name] = [p.detach().float().clone() for p in arms[name]["model"].parameters()]
    worst = max(((a - b).abs() / (b.abs() + 1e-2)).max().item() for a, b in zip(check["fused_clip"],
                                                                                  check["unfused_clip"]))
    # torch returns the norm of bf16 gradients in bf16
    norms = (arms["fused_clip"]["opt"].grad_norm().item(), arms["unfused_clip"]["opt"].grad_norm().item())
    del check

    # ---- capture every arm, then alternate timed windows
    graphs = {}
    for name, arm in arms.items():
        warm = 11 if arm["fused"] is None else 3
        pre = arm["opt"].refresh_hparams if arm["fused"] else None
        graphs[name] = GraphedStep(step_fn(arm), warmup=warm, pre_replay=pre, device=device)
        sync_all()
    ms = {n: [] for n in arms}
    exposed = {n: [] for n in arms}
    for _ in range(args.rounds):
        for name, g in graphs.items():
            for _ in range(args.warmup):
                g()
            sync_all()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                g()
            e1.record()
            torch.cuda.synchronize(device)
            t = e0.elapsed_time(e1) / args.steps
            if world > 1:
                tt = torch.tensor([t], device=device)
                torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
                t = tt.item()
            ms[name].append(t)
            gs = getattr(arms[name]["opt"], "grad_sync", None)
            if gs is not None:
                exposed[name].append(gs.exposed_comm_ms())
            sync_all()
    name_gpu, power = gpu_info(torch, device)
    if rank == 0:
        med = {n: statistics.median(v) for n, v in ms.items()}
        res = {
            "workload": "bert_large bf16 AdamW, per-GPU batch %d x seq %d, whole step graph-captured" % (B, S),
            "gpus": world, "gpu": name_gpu, "power_limit_w": power, "max_grad_norm": mn,
            "ms_per_step": {n: round(v, 3) for n, v in med.items()},
            "ms_per_step_rounds": {n: [round(x, 3) for x in v] for n, v in ms.items()},
            "exposed_comm_ms": {n: (None if not v or v[-1] is None else round(v[-1], 3)) for n, v in exposed.items()},
            "clip_cost_ms": round(med["fused_clip"] - med["fused"], 3),
            "clip_cost_pct": round(100.0 * (med["fused_clip"] / med["fused"] - 1.0), 2),
            "fused_clip_vs_ddp_clip": (round(med["ddp_clip"] / med["fused_clip"], 3) if "ddp_clip" in med else None),
            "check": {"steps": args.check_steps, "max_rel_param_diff_fused_vs_unfused": worst,
                      "grad_norm_fused_unfused": norms,
                      # two bf16 ulps on the weights, the bf16 rounding of torch's norm on the norm
                      "ok": worst < 1.6e-2 and abs(norms[0] - norms[1]) <= 1e-2 * norms[1]},
        }
        print(json.dumps(res))
    sync_all()
    if world > 1:
        sys.stdout.flush()
        os._exit(0)      # captured NCCL graphs make process-group teardown block (see bench.py)
    bps.shutdown()
    return 0


if __name__ == "__main__":
    sys.exit(main())
