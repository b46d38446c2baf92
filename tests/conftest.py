import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


@pytest.fixture(scope="session")
def lib():
    """libhectorb200.so, built in-tree if needed (nvcc cross-compiles without a GPU)."""
    from isaac_b200 import _lib, build
    build.build()
    return _lib.load()


@pytest.fixture(scope="session")
def cuda_device():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


from oracle.ref_harness import reference_root  # noqa: E402

HAVE_REFERENCE = reference_root() is not None      # the upstream source (oracle/ref_harness.py)
