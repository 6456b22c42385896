import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    """`pytest tests` on a box without a CUDA device (or without the built library) skips the gpu-marked tests instead
    of failing every one of them in Engine.__init__."""
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    if have_gpu:
        return          # with a GPU present a missing libalq.so must FAIL the gpu tests, not skip them
    skip = pytest.mark.skip(reason="gpu test: no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def gold():
    from helpers import load_gold
    return load_gold()
