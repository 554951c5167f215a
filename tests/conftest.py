import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch

    has_gpu = torch.cuda.is_available()
    for it in items:
        if "gpu" in it.keywords and not has_gpu:
            it.add_marker(pytest.mark.skip(reason="no CUDA device"))
