import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
os.environ.setdefault("DSB200_LOG_LEVEL", "warning")
os.environ.setdefault("MASTER_ADDR", "127.0.0.1")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "world_size(n): number of ranks for a distributed test")
    config.addinivalue_line("markers", "slow: long-running test")


@pytest.fixture(autouse=True)
def _host_tier_unless_marked_gpu(request, monkeypatch):
    """Tests not marked ``gpu`` are the host tier (CPU tensors, gloo): on a machine with a GPU they run as on one without,
    in this process (``torch.cuda.is_available()`` is False, host accelerator, a process group a GPU test left open is
    closed) and in every process they start (no visible device)."""
    import torch
    if "gpu" in request.node.keywords or not torch.cuda.is_available():
        yield
        return
    import torch.distributed as dist
    from deepspeed_b200 import comm
    from deepspeed_b200.accelerator import set_accelerator
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    if dist.is_initialized() and dist.get_backend() != "gloo":
        comm.destroy_process_group()
    set_accelerator(None)  # chosen again on next use
    yield
    set_accelerator(None)


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="needs a CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)
