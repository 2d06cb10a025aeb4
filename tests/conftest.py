import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu under gpurun)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture
def recorded_threads():
    """Run on the 8 torch intra-op threads the bit-exact CPU fixtures were recorded with (on an AVX-512 host).  oneDNN
    splits fp32 convolution sums by thread count, so a replay on another count differs in the last bits."""
    import torch
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)
