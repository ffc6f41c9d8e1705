"""Global-norm gradient clipping inside the fused optimizer exchange (kernels/pushpull_clip.cu).

Kernel level on `VirtualCluster` (N virtual ranks on one GPU), the public API on one GPU, and real multi-process runs
(>= 2 GPUs)."""
import os
import struct

import pytest
import torch

from _mp import run_workers

pytestmark = pytest.mark.gpu

DT = {"f32": torch.float32, "bf16": torch.bfloat16}
SIZES = [8 * 1031, 8 * 37, 8 * 5003]      # bucket element counts; none is a multiple of 8 x world for world > 1
GROUP = [0, 0, 1]                          # buckets 0 and 1 in param group 0, bucket 2 in group 1
LR = {"sgd": (0.1, 0.05), "adam": (0.01, 0.003)}


def _cu():
    from byteps_b200 import _native

    return _native.cuda()


def _code(dt):
    from byteps_b200.comm.symm import wire_code

    return wire_code(dt)


def _hp(kind, lr, step):
    """OptHParams blob (pushpull.cuh) of one param group."""
    if kind.startswith("sgd"):
        vals = (lr, 0.01, 0.9, 0.0, 0.9, 0.999, 1e-8, 1.0, 1.0, int(kind.endswith("nesterov")), 0, int(step == 1), 1.0)
    else:
        vals = (lr, 0.01, 0.0, 0.0, 0.9, 0.999, 1e-8, 1 - 0.9 ** step, 1 - 0.999 ** step, 0, int(kind == "adamw"),
                int(step == 1), 1.0)
    return struct.pack("<9f3if3i", *vals, 0, 0, 0)


def _ref_opt(kind, params, group=GROUP):
    lrs = LR["sgd" if kind.startswith("sgd") else "adam"]
    groups = [{"params": [p for p, g in zip(params, group) if g == gi], "lr": lrs[gi]} for gi in range(2)]
    if kind.startswith("sgd"):
        return torch.optim.SGD(groups, lr=lrs[0], momentum=0.9, weight_decay=0.01, nesterov=kind.endswith("nesterov"))
    if kind == "adam":
        return torch.optim.Adam(groups, lr=lrs[0], weight_decay=0.01)
    return torch.optim.AdamW(groups, lr=lrs[0], weight_decay=0.01)


def _run_virtual(world, dtype, kind, max_norm, steps, engine="clip", sizes=SIZES, group=GROUP,
                 update_blocks=3):
    """Buckets of `sizes` elements through the clip phases (engine="clip", phase 3 on `update_blocks` CTAs) or the
    existing fused TMA kernel (engine="fused").
    Returns per step [(state bytes of every rank, own averaged shards)], final params of every rank, fp32 masters."""
    from byteps_b200.comm.symm import VirtualCluster

    cu = _cu()
    es = torch.empty((), dtype=dtype).element_size()
    goffs, poffs, off = [], [], 0
    for n in sizes:
        goffs.append(off)
        off += (n * es + 255) // 256 * 256
    for n in sizes:
        poffs.append(off)
        off += (n * es + 255) // 256 * 256
    pub = off
    vc = VirtualCluster(world, "cuda:0", off + 4096)
    gen = torch.Generator(device="cuda").manual_seed(5)
    w0 = [torch.randn(n, device="cuda", generator=gen).to(dtype) for n in sizes]
    nstate = 2 if kind.startswith("sgd") else 3
    state = [[[] for _ in sizes] for _ in range(world)]      # [rank][bucket] -> [master, s0, s1]
    for r in range(world):
        for bi, n in enumerate(sizes):
            b, e = cu.shard_units(n // 8, world, r)
            m = torch.zeros(max((e - b) * 8, 8), device="cuda")
            m[:(e - b) * 8] = w0[bi].float()[b * 8:e * 8]
            state[r][bi] = [m] + [torch.zeros_like(m) for _ in range(nstate - 1)] + [torch.zeros_like(m)] * (3 - nstate)
            vc.arenas[r][poffs[bi]:poffs[bi] + n * es].view(dtype).copy_(w0[bi])
    # per rank: rows 0-1 the two groups' hyper-parameters, row 2 the ClipState
    hp = [torch.zeros((3, 64), dtype=torch.uint8, device="cuda") for _ in range(world)]
    slots = [torch.zeros(len(sizes) * cu.CLIP_SLOTS_PER_BUCKET, dtype=torch.float64, device="cuda")
             for _ in range(world)]
    code = cu.OPT_SGD if kind.startswith("sgd") else cu.OPT_ADAM
    tables = []
    for r in range(world):
        rows = [[goffs[bi], poffs[bi], n, state[r][bi][0].data_ptr(), state[r][bi][1].data_ptr(),
                 state[r][bi][2].data_ptr(), hp[r].data_ptr() + 64 * group[bi], 0] for bi, n in enumerate(sizes)]
        tables.append(torch.tensor(rows, dtype=torch.int64, device="cuda"))
    lrs = LR["sgd" if kind.startswith("sgd") else "adam"]
    out = []
    for step in range(1, steps + 1):
        blob = _hp(kind, lrs[0], step) + _hp(kind, lrs[1], step) + struct.pack("<f", max_norm)
        for r in range(world):
            cu.write_blob(hp[r].data_ptr(), blob, torch.cuda.current_stream().cuda_stream)
        grads = [[torch.randn(n, device="cuda", generator=gen).to(dtype) for n in sizes] for _ in range(world)]
        for r in range(world):
            for bi, n in enumerate(sizes):
                vc.arenas[r][goffs[bi]:goffs[bi] + n * es].view(dtype).copy_(grads[r][bi])
        if engine == "clip":
            for bi, n in enumerate(sizes):
                vc.run(lambda r, view, arena, s: cu.clip_reduce_sumsq(
                    view, _code(dtype), goffs[bi], n, 1.0 / world,
                    slots[r].data_ptr() + 8 * cu.CLIP_SLOTS_PER_BUCKET * bi, hp[r].data_ptr() + 64 * group[bi],
                    2 + bi % 2, 256, 0, False, s))
            vc.run(lambda r, view, arena, s: cu.clip_finalize(view, slots[r].data_ptr(), slots[r].numel(), pub,
                                                              hp[r].data_ptr() + 128, 0, s))
            vc.run(lambda r, view, arena, s: cu.clip_update(view, _code(dtype), code, tables[r].data_ptr(), len(sizes),
                                                            hp[r].data_ptr() + 128, update_blocks, 3, False, 0,
                                                            s))
        else:
            for bi, n in enumerate(sizes):
                vc.run(lambda r, view, arena, s: cu.pushpull_fused_opt_tma(
                    view, _code(dtype), code, goffs[bi], poffs[bi], n, 1.0 / world, state[r][bi][0].data_ptr(),
                    state[r][bi][1].data_ptr(), state[r][bi][2].data_ptr(), hp[r].data_ptr() + 64 * group[bi], 2, 3,
                    False, 0, s))
        torch.cuda.synchronize()
        own = []      # every bucket's averaged gradient as phase 1 wrote it, assembled from the owners' shards
        for bi, n in enumerate(sizes):
            parts = []
            for r in range(world):
                b, e = cu.shard_units(n // 8, world, r)
                parts.append(vc.arenas[r][goffs[bi]:goffs[bi] + n * es].view(dtype)[b * 8:e * 8].clone())
            own.append(torch.cat(parts))
        out.append(([hp[r][2, :16].clone() for r in range(world)], own, grads))
    params = [[vc.arenas[r][poffs[bi]:poffs[bi] + n * es].view(dtype).clone() for bi, n in enumerate(sizes)]
              for r in range(world)]
    masters = []
    for bi, n in enumerate(sizes):
        parts = []
        for r in range(world):
            b, e = cu.shard_units(n // 8, world, r)
            parts.append(state[r][bi][0][:(e - b) * 8])
        masters.append(torch.cat(parts))
    return out, params, masters, w0


@pytest.mark.parametrize("world", [1, 2, 4, 8])
@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("kind", ["sgd", "sgd_nesterov", "adam", "adamw"])
@pytest.mark.parametrize("active", [True, False])
def test_clip_kernels_virtual(world, dt, kind, active):
    dtype = DT[dt]
    max_norm = 1.0 if active else 1e6     # the averaged gradients' norm is ~220 / sqrt(world)
    steps = 3
    out, params, masters, w0 = _run_virtual(world, dtype, kind, max_norm, steps)
    ref_p = [torch.nn.Parameter(w.float().clone()) for w in w0]
    ropt = _ref_opt(kind, ref_p)
    for states, own, grads in out:
        # norm and coefficient bit-identical on every virtual rank
        for s in states[1:]:
            assert torch.equal(s[4:12], states[0][4:12])
        norm, coef = states[0][4:12].view(torch.float32).tolist()
        ref_norm = torch.sqrt(sum((g.double() ** 2).sum() for g in own)).item()
        assert abs(norm - ref_norm) <= 1e-6 * ref_norm, (norm, ref_norm)
        assert (coef < 1.0) == active
        # what phase 1 wrote is the average of the ranks' gradients
        for bi, g in enumerate(own):
            avg = torch.stack([grads[r][bi].float() for r in range(world)]).sum(0) / world
            tol = 1e-6 if dtype == torch.float32 else 8e-3
            assert torch.allclose(g.float(), avg, atol=tol, rtol=tol)
        # the reference clips and steps on the averaged gradients as exchanged (bf16: rounded once): with Adam's L2
        # weight decay competing with a clipped gradient, the rounding alone can flip the sign of an update
        for p, g in zip(ref_p, own):
            p.grad = g.float()
        tn = torch.nn.utils.clip_grad_norm_(ref_p, max_norm)
        assert abs(tn.item() - norm) <= 1e-5 * norm
        ropt.step()
    tol_p = 1e-5 if dtype == torch.float32 else 1.2e-2
    tol_m = 1e-5 if dtype == torch.float32 else 2e-2
    for r in range(world):
        for bi in range(len(SIZES)):
            assert torch.equal(params[r][bi], params[0][bi])
            got = params[r][bi].float()
            assert torch.allclose(got, ref_p[bi].detach(), atol=tol_p, rtol=tol_p), \
                (r, bi, (got - ref_p[bi].detach()).abs().max())
    for bi in range(len(SIZES)):
        assert torch.allclose(masters[bi], ref_p[bi].detach(), atol=tol_m, rtol=tol_m), \
            (bi, (masters[bi] - ref_p[bi].detach()).abs().max())
    # run to run: the same inputs give bit-identical norms, coefficients and parameters
    out2, params2, _, _ = _run_virtual(world, dtype, kind, max_norm, steps)
    for (s1, _, _), (s2, _, _) in zip(out, out2):
        assert torch.equal(s1[0][4:12], s2[0][4:12])
    for bi in range(len(SIZES)):
        assert torch.equal(params2[0][bi], params[0][bi])
    if dtype == torch.float32 and not active:
        # inactive clipping computes what the fused exchange computes
        _, fparams, fmasters, _ = _run_virtual(world, dtype, kind, max_norm, steps, engine="fused")
        for bi in range(len(SIZES)):
            assert torch.allclose(params[0][bi], fparams[0][bi], atol=1e-6, rtol=1e-6)
            assert torch.allclose(masters[bi], fmasters[bi], atol=1e-6, rtol=1e-6)


@pytest.mark.parametrize("world", [2, 8])
@pytest.mark.parametrize("kind", ["sgd", "adamw"])
def test_clip_update_grid_is_rank_independent(world, kind):
    """Phase 3 ends in a barrier between the CTAs of equal index on every rank, so every rank must launch the same
    grid.  Here the ranks own different numbers of tiles (the last shards are shorter, one is empty at 8 ranks), and
    the kernels run with the grid BucketedGradSync computes."""
    from byteps_b200.parallel.bucket import clip_update_grid

    cu = _cu()
    sizes, group = [8 * 1025, 8 * 9], [0, 1]
    tiles = []
    for r in range(world):
        t = 0
        for n in sizes:
            b, e = cu.shard_units(n // 8, world, r)
            t += ((e - b) * 8 * 4 // 16 + 255) // 256
        tiles.append(t)
    assert len(set(tiles)) > 1, tiles
    grid = clip_update_grid(sizes, 4, world)
    assert grid == max(tiles)
    out, params, masters, w0 = _run_virtual(world, torch.float32, kind, 1.0, 3, sizes=sizes, group=group,
                                            update_blocks=grid)
    ref_p = [torch.nn.Parameter(w.float().clone()) for w in w0]
    ropt = _ref_opt(kind, ref_p, group)
    for states, own, _ in out:
        for s in states[1:]:
            assert torch.equal(s[4:12], states[0][4:12])
        for p, g in zip(ref_p, own):
            p.grad = g.float()
        torch.nn.utils.clip_grad_norm_(ref_p, 1.0)
        ropt.step()
    for r in range(world):
        for bi in range(len(sizes)):
            assert torch.equal(params[r][bi], params[0][bi])
            assert torch.allclose(params[r][bi], ref_p[bi].detach(), atol=1e-5, rtol=1e-5)
    for bi in range(len(sizes)):
        assert torch.allclose(masters[bi], ref_p[bi].detach(), atol=1e-5, rtol=1e-5)


# ---------------------------------------------------------------- public API, one GPU
class _Net(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.l1 = torch.nn.Linear(37, 29)       # 1073 + 29 elements: padded inside the bucket
        self.l2 = torch.nn.Linear(29, 10)       # a bias of 10 elements
        self.unused = torch.nn.Parameter(torch.randn(13))

    def forward(self, x):
        return self.l2(torch.relu(self.l1(x)))


def _pair(opt_name, **kw):
    torch.manual_seed(11)
    m1, m2 = _Net().cuda(), _Net().cuda()
    m2.load_state_dict(m1.state_dict())
    groups = lambda m: [{"params": [m.l1.weight, m.l1.bias, m.unused]}, {"params": list(m.l2.parameters()),  # noqa: E731
                                                                         "lr": 0.02 if opt_name == "sgd" else 3e-3}]
    if opt_name == "sgd":
        mk = lambda m: torch.optim.SGD(groups(m), lr=0.05, momentum=0.9)  # noqa: E731
    else:
        mk = lambda m: torch.optim.AdamW(groups(m), lr=1e-2, weight_decay=0.01)  # noqa: E731
    return m1, m2, mk(m1), mk(m2)


def _ref_step(m, opt, x, y, max_norm):
    opt.zero_grad()
    torch.nn.functional.cross_entropy(m(x), y).backward()
    for p in m.parameters():
        if p.grad is None:
            p.grad = torch.zeros_like(p)     # unused this step: the fused exchange counts it as a zero gradient
    n = torch.nn.utils.clip_grad_norm_(list(m.parameters()), max_norm)
    opt.step()
    return n


@pytest.mark.parametrize("opt_name", ["sgd", "adamw"])
@pytest.mark.parametrize("graph", [False, True])
def test_distributed_optimizer_clip_one_gpu(opt_name, graph):
    import byteps_b200.torch as bps
    from byteps_b200.torch.graph import GraphedStep

    bps.init()
    m1, m2, inner, ropt = _pair(opt_name)
    opt = bps.DistributedOptimizer(inner, named_parameters=m1.named_parameters(), fused_update=True, max_grad_norm=0.5)
    assert opt.grad_sync.clip and opt.grad_sync._ring_mode == "off"
    torch.manual_seed(12)
    xs = torch.randn(8, 16, 37, device="cuda")
    ys = torch.randint(0, 10, (8, 16), device="cuda")
    sx, sy = torch.empty(16, 37, device="cuda"), torch.empty(16, dtype=torch.long, device="cuda")

    def step():
        opt.zero_grad()
        torch.nn.functional.cross_entropy(m1(sx), sy).backward()
        opt.step()

    runner = None
    # (max_grad_norm, lr factor) per step: clipping active, then inactive, then active again.  The lr schedule runs
    # under the graph only: eager fused steps publish a group's hyper-parameters at the end of the previous step.
    plan = [(0.5, 1.0), (0.5, 1.0), (0.5, 1.0), (0.5, 1.0), (100.0, 1.0), (100.0, 0.5), (0.2, 0.5), (0.2, 0.25)]
    if not graph:
        plan = [(mn, 1.0) for mn, _ in plan]
    base = [g["lr"] for g in opt.param_groups]
    norms = []
    for i, (mn, f) in enumerate(plan):
        sx.copy_(xs[i])
        sy.copy_(ys[i])
        for g, g2, b in zip(opt.param_groups, ropt.param_groups, base):
            g["lr"] = g2["lr"] = b * f
        if opt.max_grad_norm != mn:
            opt.max_grad_norm = mn
        if graph and i >= 2:
            if runner is None:
                runner = GraphedStep(step, warmup=1, pre_replay=opt.refresh_hparams)   # runs this batch eagerly
            else:
                runner()
        else:
            step()
        rn = _ref_step(m2, ropt, sx, sy, mn)
        torch.cuda.synchronize()
        norms.append((opt.grad_norm().item(), rn.item(), mn))
    assert opt.grad_norm().dim() == 0 and opt.grad_norm().dtype == torch.float32 and opt.grad_norm().is_cuda
    for got, want, mn in norms:
        assert abs(got - want) <= 1e-5 * max(1.0, want), norms
    assert any(want > mn for _, want, mn in norms) and any(want < mn for _, want, mn in norms), norms
    for a, b in zip(m1.parameters(), m2.parameters()):
        assert torch.allclose(a, b, atol=1e-5), (a - b).abs().max()
    bps.shutdown()


def test_clip_nan_gradient_matches_torch():
    import byteps_b200.torch as bps

    bps.init()
    m1, m2, inner, ropt = _pair("sgd")
    opt = bps.DistributedOptimizer(inner, named_parameters=m1.named_parameters(), fused_update=True, max_grad_norm=1.0)
    x = torch.randn(4, 37, device="cuda")
    x[1, 3] = float("nan")
    y = torch.randint(0, 10, (4,), device="cuda")
    opt.zero_grad()
    torch.nn.functional.cross_entropy(m1(x), y).backward()
    opt.step()
    rn = _ref_step(m2, ropt, x, y, 1.0)
    torch.cuda.synchronize()
    assert torch.isnan(opt.grad_norm()).item() and torch.isnan(rn).item()
    for a, b in zip(m1.parameters(), m2.parameters()):
        assert torch.equal(torch.isnan(a), torch.isnan(b))
        assert torch.allclose(a[~torch.isnan(a)], b[~torch.isnan(b)], atol=1e-5)
    bps.shutdown()


def test_half_precision_clip_norm_is_unscaled():
    import byteps_b200.torch as bps
    from byteps_b200.torch.half_optimizer import HalfPrecisionDistributedOptimizer

    bps.init()
    torch.manual_seed(13)
    m1 = _Net().cuda().to(torch.bfloat16)
    m2 = _Net().cuda().to(torch.bfloat16)
    m2.load_state_dict(m1.state_dict())
    opt = HalfPrecisionDistributedOptimizer(torch.optim.SGD(m1.parameters(), lr=0.05, momentum=0.9),
                                            named_parameters=m1.named_parameters(), loss_scale=1024.0,
                                            max_grad_norm=0.7)
    assert opt.max_grad_norm == 0.7
    opt.max_grad_norm = 0.3             # reaches the fused exchange through the wrapped optimizer
    assert opt.max_grad_norm == 0.3 and opt.grad_sync.max_grad_norm == 0.3
    x = torch.randn(16, 37, device="cuda").to(torch.bfloat16)
    y = torch.randint(0, 10, (16,), device="cuda")
    opt.zero_grad()
    opt.backward(torch.nn.functional.cross_entropy(m1(x).float(), y))
    opt.step()
    (torch.nn.functional.cross_entropy(m2(x).float(), y) * 1024.0).backward()
    want = torch.sqrt(sum((p.grad.double() / 1024.0).pow(2).sum() for p in m2.parameters() if p.grad is not None))
    torch.cuda.synchronize()
    got = opt.grad_norm().item()
    assert abs(got - want.item()) <= 1e-3 * want.item(), (got, want.item())
    assert want.item() > 0.3        # clipping was active
    bps.shutdown()


def test_fused_clip_rejects_wire_cast():
    import byteps_b200.torch as bps

    bps.init()
    m = _Net().cuda()
    with pytest.raises(ValueError, match="wire cast"):
        bps.DistributedOptimizer(torch.optim.SGD(m.parameters(), lr=0.1), named_parameters=m.named_parameters(),
                                 compression=bps.Compression.fp16, fused_update=True, max_grad_norm=1.0)
    bps.shutdown()


# ---------------------------------------------------------------- several GPUs
def _multi(rank, world, outdir, graph):
    import byteps_b200.torch as bps
    from byteps_b200.torch.graph import GraphedStep

    torch.cuda.set_device(rank)
    bps.init()
    torch.manual_seed(100 + rank)
    mk = lambda: torch.nn.Sequential(torch.nn.Linear(61, 133), torch.nn.ReLU(), torch.nn.Linear(133, 10)).cuda()  # noqa: E731
    model = mk()
    opt = bps.DistributedOptimizer(torch.optim.AdamW(model.parameters(), lr=1e-2, weight_decay=0.01),
                                   named_parameters=model.named_parameters(), fused_update=True, max_grad_norm=0.5)
    assert opt.grad_sync._ring_mode == "off"
    bps.broadcast_parameters(model.state_dict(), root_rank=0)
    ref = mk()
    ref.load_state_dict(model.state_dict())
    ropt = torch.optim.AdamW(ref.parameters(), lr=1e-2, weight_decay=0.01)
    torch.manual_seed(7)
    steps = 6
    xs = torch.randn(steps, world * 8, 61, device="cuda")
    ys = torch.randint(0, 10, (steps, world * 8), device="cuda")
    sx, sy = torch.empty(8, 61, device="cuda"), torch.empty(8, dtype=torch.long, device="cuda")

    def step():
        opt.zero_grad()
        torch.nn.functional.cross_entropy(model(sx), sy).backward()
        opt.step()

    runner, norms = None, []
    for i in range(steps):
        sx.copy_(xs[i, rank * 8:(rank + 1) * 8])
        sy.copy_(ys[i, rank * 8:(rank + 1) * 8])
        if graph and i >= 2:
            if runner is None:
                runner = GraphedStep(step, warmup=1, pre_replay=opt.refresh_hparams)
            else:
                runner()
        else:
            step()
        ropt.zero_grad()
        torch.nn.functional.cross_entropy(ref(xs[i]), ys[i]).backward()   # full batch = mean of the rank means
        rn = torch.nn.utils.clip_grad_norm_(list(ref.parameters()), 0.5)
        ropt.step()
        torch.cuda.synchronize()
        norms.append(opt.grad_norm().item())
        assert abs(norms[-1] - rn.item()) <= 1e-4 * rn.item(), (i, norms[-1], rn.item())
    for a, b in zip(model.parameters(), ref.parameters()):
        assert torch.allclose(a, b, atol=1e-4), (a - b).abs().max()
    torch.save({"params": [p.detach().cpu() for p in model.parameters()], "norms": norms},
               os.path.join(outdir, "rank%d.pt" % rank))
    bps.shutdown()


def _worlds():
    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    return [2] + ([n] if n >= 4 else [])


@pytest.mark.multigpu
@pytest.mark.parametrize("env", ["nvls_auto", "nvls_off", "ring_batch"])
@pytest.mark.parametrize("graph", [False, True])
def test_fused_clip_multi_gpu(env, graph, tmp_path):
    extra = {"nvls_auto": {}, "nvls_off": {"BYTEPS_USE_NVLS": "0"}, "ring_batch": {"BYTEPS_RING": "batch"}}[env]
    for world in _worlds():
        d = tmp_path / ("w%d" % world)
        d.mkdir()
        run_workers(_multi, world=world, args=(str(d), graph), env=extra, timeout=300)
        outs = [torch.load(d / ("rank%d.pt" % r)) for r in range(world)]
        for o in outs[1:]:
            assert o["norms"] == outs[0]["norms"]          # bit-identical floats
            for a, b in zip(o["params"], outs[0]["params"]):
                assert torch.equal(a, b)
