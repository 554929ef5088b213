import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line(
        "markers", "reference: runs the original VMAS project's own files (VMAS_REF: its checkout; else oracle/_ref)"
    )


def pytest_collection_modifyitems(config, items):
    import torch

    from refutil import have_reference

    has_gpu = torch.cuda.is_available()
    has_ref = have_reference()
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "reference" in item.keywords and not has_ref:
            item.add_marker(pytest.mark.skip(reason="reference checkout not present"))
