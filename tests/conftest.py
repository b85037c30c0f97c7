import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def port():
    from oracle import loader
    if not loader.available("port"):
        loader.build(("port",))
    return loader.Oracle("port")


@pytest.fixture(scope="session")
def oracle(request):
    """Best available checker: the compiled reference if present, else the port."""
    from oracle import loader
    if loader.available("reference"):
        return loader.Oracle("reference")
    if not loader.available("port"):
        loader.build(("port",))
    return loader.Oracle("port")


@pytest.fixture(scope="session")
def engine():
    """The CUDA engine through its C ABI; never falls back to anything else."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from bayeslogit_b200 import _lib, api
    _lib.lib()
    return api
