import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "friendly-stable-audio-tools_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


def pytest_collection_modifyitems(config, items):
    import torch
    has_cuda = torch.cuda.is_available()
    for item in items:
        if "gpu" in item.keywords and not has_cuda:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN
