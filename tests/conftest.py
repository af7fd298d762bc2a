import importlib.util
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def pytest_collection_modifyitems(config, items):
    """On a box without a CUDA device the gpu-marked tests are skipped instead of erroring (a plain `pytest` is green there);
    on the GPU box nothing is skipped - a missing libvfi_b200.so still fails loudly, by design."""
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    if have_gpu:
        return
    skip = pytest.mark.skip(reason="needs a B200 (torch.cuda.is_available() is False)")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


def load_pkg():
    """Import the product package (its directory name has a hyphen, like every ComfyUI custom node)."""
    import __graft_entry__ as ge
    return ge.load_package()


@pytest.fixture(scope="session")
def pkg():
    return load_pkg()


GOLDEN_CPU_THREADS = 8


@pytest.fixture
def golden_cpu_threads():
    """The reference outputs in tests/golden were made on the CPU with 8 intra-op threads.  ATen splits some fp32
    reductions by thread count, so the oracle meets them at rounding level only when it runs with the same count."""
    import torch
    before = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_CPU_THREADS)
    yield
    torch.set_num_threads(before)
