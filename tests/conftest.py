import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA sm_100 device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: runs the unmodified reference itself; skips unless its source tree is found (oracle/refload.py)")


def pytest_collection_modifyitems(config, items):
    import torch
    has_gpu = torch.cuda.is_available()
    skip_gpu = pytest.mark.skip(reason="no CUDA device")
    from oracle import refload
    skip_ref = pytest.mark.skip(reason="reference tree not present")
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(skip_gpu)
        if "reference" in item.keywords and not refload.available():
            item.add_marker(skip_ref)


@pytest.fixture(scope="session")
def built_lib():
    from novic_b200 import _abi
    if not os.path.isfile(_abi.LIB_PATH):
        _abi.build()
    return _abi.lib()
