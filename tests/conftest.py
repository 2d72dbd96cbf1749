import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden(name):
    return torch.load(os.path.join(GOLDEN, name), map_location="cpu", weights_only=False)


@pytest.fixture
def golden_threads():
    """Bit-exact CPU comparisons with the goldens run with the intra-op thread count the goldens were made with: torch's
    fp32 CPU kernels split their sums by it, so the last bits depend on it.  Restored afterwards."""
    from oracle.make_golden import CPU_THREADS
    prev = torch.get_num_threads()
    torch.set_num_threads(CPU_THREADS)
    yield
    torch.set_num_threads(prev)


@pytest.fixture
def emu():
    """Install the torch emulation of the ops interface (host-logic tests on CPU), restore afterwards."""
    import minimagen_b200.ops as ops_mod
    from emu_ops import EmuOps
    prev = ops_mod._OPS
    e = EmuOps()
    ops_mod.set_ops(e)
    yield e
    ops_mod.set_ops(prev)


@pytest.fixture
def native():
    """The real backend (GPU tests).  Fails -- not skips -- if the library is missing on a GPU box."""
    import minimagen_b200.ops as ops_mod
    from minimagen_b200 import _native
    _native.load()
    prev = ops_mod._OPS
    ops_mod.set_ops(ops_mod.NativeOps())
    yield ops_mod._OPS
    ops_mod.set_ops(prev)


def rel_l2(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / b.norm().clamp(min=1e-30)).item()
