import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_report_header(config):
    import ref_harness
    if ref_harness.ref_module() is not None:
        return "parity reference: the reference CUDA extension (oracle/_ref)"
    return ("parity reference: the CPU oracle, checked against the recorded reference outputs "
            "(tests/golden/parity_record.npz); the reference CUDA extension oracle/_ref is not built")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)
