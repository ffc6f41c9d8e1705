#!/usr/bin/env python
"""BERT-large pre-training step loop (the reference's bandwidth-bound headline
workload) with the fused Adam exchange: bf16 parameters/gradients, fp32 master
weights and moments sharded over the GPUs, one kernel per bucket."""
import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
import byteps_b200.torch as bps  # noqa: E402
from byteps_b200.models import get_model  # noqa: E402

p = argparse.ArgumentParser()
p.add_argument("--model", default="bert_large")
p.add_argument("--batch-size", type=int, default=16)
p.add_argument("--seq-len", type=int, default=128)
p.add_argument("--steps", type=int, default=20)
p.add_argument("--warmup-steps", type=int, default=5)
p.add_argument("--no-cuda", action="store_true", help="CPU run over gloo (unfused optimizer, fp32)")
p.add_argument("--max-grad-norm", type=float, default=None,
               help="clip the averaged gradients to this global L2 norm every step (default: no clipping)")
args = p.parse_args()
bps.init()
cuda = torch.cuda.is_available() and not args.no_cuda
if cuda:
    torch.cuda.set_device(bps.local_rank())
dev = torch.device("cuda", bps.local_rank()) if cuda else torch.device("cpu")
model = get_model(args.model).to(dev)
if cuda:
    model = model.to(torch.bfloat16)
opt = bps.DistributedOptimizer(torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.01),
                               named_parameters=model.named_parameters(), fused_update=cuda,
                               max_grad_norm=args.max_grad_norm)
bps.broadcast_parameters(model.state_dict(), root_rank=0)
ids = torch.randint(0, 30522, (args.batch_size, args.seq_len), device=dev)
labels = torch.randint(0, 30522, (args.batch_size, args.seq_len), device=dev)


def sync():
    if cuda:
        torch.cuda.synchronize()


for i in range(args.steps + args.warmup_steps):
    if i == args.warmup_steps:
        sync()
        t0 = time.time()
    opt.zero_grad()
    loss = model(ids, mlm_labels=labels)
    loss.backward()
    opt.step()
sync()
if bps.rank() == 0:
    dt = time.time() - t0
    print("tokens/sec on %d %s(s): %.0f (loss %.3f)" % (bps.size(), "GPU" if cuda else "CPU worker",
                                                         bps.size() * args.batch_size * args.seq_len * args.steps / dt,
                                                         loss.item()))
bps.shutdown()
