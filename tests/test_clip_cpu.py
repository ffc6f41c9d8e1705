"""max_grad_norm on the CPU paths: clip_grad_norm_ between the gradient exchange and the wrapped optimizer's step, and
the arguments the option refuses."""
import math
import types

import pytest
import torch

from _mp import run_workers


def _gloo_clip(rank, world):
    import byteps_b200.torch as bps

    bps.init()
    torch.manual_seed(1234 + rank)
    model = torch.nn.Sequential(torch.nn.Linear(8, 16), torch.nn.ReLU(), torch.nn.Linear(16, 4))
    opt = bps.DistributedOptimizer(torch.optim.SGD(model.parameters(), lr=0.1, momentum=0.9),
                                   named_parameters=model.named_parameters(), max_grad_norm=0.25)
    assert opt.grad_norm() is None
    bps.broadcast_parameters(model.state_dict(), root_rank=0)
    bps.broadcast_optimizer_state(opt, root_rank=0)
    ref = torch.nn.Sequential(torch.nn.Linear(8, 16), torch.nn.ReLU(), torch.nn.Linear(16, 4))
    ref.load_state_dict(model.state_dict())
    ref_opt = torch.optim.SGD(ref.parameters(), lr=0.1, momentum=0.9)
    torch.manual_seed(99)
    clipped = 0
    for i in range(4):
        x, y = torch.randn(world * 4, 8), torch.randn(world * 4, 4) * 5
        if i == 2:
            opt.max_grad_norm = 1e3      # inactive from here on
        opt.zero_grad()
        torch.nn.functional.mse_loss(model(x[rank * 4:(rank + 1) * 4]), y[rank * 4:(rank + 1) * 4]).backward()
        opt.step()
        ref_opt.zero_grad()
        torch.nn.functional.mse_loss(ref(x), y).backward()
        n = torch.nn.utils.clip_grad_norm_(list(ref.parameters()), opt.max_grad_norm)
        ref_opt.step()
        clipped += int(n.item() > opt.max_grad_norm)
        assert abs(opt.grad_norm().item() - n.item()) <= 1e-5 * n.item()
    assert clipped == 2
    for a, b in zip(model.parameters(), ref.parameters()):
        assert torch.allclose(a, b, atol=1e-5), (a - b).abs().max()
    bps.shutdown()


def test_gloo_unfused_path_clips_like_torch():
    run_workers(_gloo_clip, world=2)


@pytest.mark.parametrize("bad", [0, -1.0, math.inf, math.nan])
def test_max_grad_norm_must_be_finite_and_positive(bad):
    import byteps_b200.torch as bps

    m = torch.nn.Linear(4, 4)
    with pytest.raises(ValueError, match="max_grad_norm"):
        bps.DistributedOptimizer(torch.optim.SGD(m.parameters(), lr=0.1), named_parameters=m.named_parameters(),
                                 max_grad_norm=bad)


def test_max_grad_norm_is_refused_in_async_mode(monkeypatch):
    import byteps_b200.torch as bps

    monkeypatch.setenv("BYTEPS_ENABLE_ASYNC", "1")
    m = torch.nn.Linear(4, 4)
    with pytest.raises(ValueError, match="BYTEPS_ENABLE_ASYNC"):
        bps.DistributedOptimizer(torch.optim.SGD(m.parameters(), lr=0.1), named_parameters=m.named_parameters(),
                                 max_grad_norm=1.0)


def test_fused_clip_refuses_a_wire_cast_of_fp32_gradients():
    from byteps_b200.parallel.bucket import BucketedGradSync

    m = torch.nn.Linear(4, 4)
    for wire in (torch.float16, torch.bfloat16):
        with pytest.raises(ValueError, match="wire cast"):
            BucketedGradSync(types.SimpleNamespace(size=2, rank=0), [{"params": list(m.parameters())}], fused="adam",
                             wire_dtype=wire, max_grad_norm=1.0)


def _half_dynamic_clip(rank, world):
    import byteps_b200.torch as bps
    from byteps_b200.torch.half_optimizer import HalfPrecisionDistributedOptimizer

    bps.init()
    torch.manual_seed(5)
    model = torch.nn.Linear(8, 4)
    ref = torch.nn.Linear(8, 4)
    ref.load_state_dict(model.state_dict())
    opt = HalfPrecisionDistributedOptimizer(torch.optim.SGD(model.parameters(), lr=0.1),
                                            named_parameters=model.named_parameters(), loss_scale=8.0,
                                            dynamic_loss_scale=True, max_grad_norm=0.1)
    assert opt.max_grad_norm == 0.1
    opt.max_grad_norm = 0.05
    assert opt.max_grad_norm == 0.05
    with pytest.raises(ValueError):
        opt.max_grad_norm = None
    with pytest.raises(ValueError):
        opt.max_grad_norm = -1.0
    x, y = torch.randn(16, 8), torch.randn(16, 4) * 10
    opt.zero_grad()
    opt.backward(torch.nn.functional.mse_loss(model(x), y))
    opt.step()
    torch.nn.functional.mse_loss(ref(x), y).backward()
    n = torch.nn.utils.clip_grad_norm_(list(ref.parameters()), 0.05)
    assert n.item() > 0.05                                 # clipping was active, with the changed value
    assert abs(opt.grad_norm().item() - n.item()) <= 1e-5 * n.item()
    with torch.no_grad():
        for p in ref.parameters():
            p -= 0.1 * p.grad
    for a, b in zip(model.parameters(), ref.parameters()):
        assert torch.allclose(a, b, atol=1e-6), (a - b).abs().max()
    bps.shutdown()


def test_half_precision_dynamic_scale_max_grad_norm_can_change():
    run_workers(_half_dynamic_clip, world=1)
