import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(autouse=True)
def _default_dtype_guard():
    prev = torch.get_default_dtype()
    yield
    torch.set_default_dtype(prev)


def relerr(a: torch.Tensor, b: torch.Tensor) -> float:
    """max |a-b| / max |b| with b the reference."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    den = max(b.abs().max().item(), 1e-30)
    return (a - b).abs().max().item() / den


def load_golden(name):
    from oracle.make_golden import expand
    return expand(torch.load(os.path.join(GOLDEN, name), weights_only=False))
