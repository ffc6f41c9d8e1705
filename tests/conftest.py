import os
import sys
import tempfile

import pytest

# VirtualCluster tests run up to 8 mutually-waiting kernels on 8 streams of one GPU: give every
# stream its own hardware queue so none is serialised behind a spinning peer (default is 8 queues).
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "multigpu: test needs >= 2 CUDA devices")


def pytest_collection_modifyitems(config, items):
    import torch

    has_gpu = torch.cuda.is_available()
    ngpu = torch.cuda.device_count() if has_gpu else 0
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "multigpu" in item.keywords and ngpu < 2:
            item.add_marker(pytest.mark.skip(reason="needs >= 2 GPUs"))


@pytest.fixture(autouse=True)
def _no_gpu_for_cpu_tests(request, monkeypatch):
    """A test without the gpu mark checks the CPU path: the processes it starts see no GPU, as on a machine without
    one.  (On a one-GPU machine its ranks would otherwise all take cuda:0, and NCCL refuses ranks that share a
    device.)"""
    if request.node.get_closest_marker("gpu") is None:
        monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")


@pytest.fixture
def sock_dir():
    """A short directory for Unix-domain sockets: a socket path holds at most 107 bytes, which tmp_path under a
    long TMPDIR can exceed."""
    with tempfile.TemporaryDirectory(prefix="bps", dir="/tmp") as d:
        yield d
