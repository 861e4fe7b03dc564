import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    for item in items:
        if "gpu" in item.keywords and not have_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
