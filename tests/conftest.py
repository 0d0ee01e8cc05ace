import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from __graft_entry__ import load_package  # noqa: E402

load_package()


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on a B200)")


def pytest_collection_modifyitems(config, items):
    """A plain ``pytest tests`` on a machine without a GPU skips the gpu-marked tests instead of failing them; with a
    GPU they run, and fail if ``__graft_entry__.build()`` has not built the library."""
    import pytest
    import torch
    if not torch.cuda.is_available():
        skip = pytest.mark.skip(reason="needs a CUDA device")
        for item in items:
            if "gpu" in item.keywords:
                item.add_marker(skip)
