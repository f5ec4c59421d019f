import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: needs a checkout of the reference at $NPI_REFERENCE_ROOT or oracle/_ref")


def pytest_collection_modifyitems(config, items):
    import torch
    has_gpu = torch.cuda.is_available()
    from oracle import ref_import
    has_ref = ref_import.reference_available()
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "reference" in item.keywords and not has_ref:
            item.add_marker(pytest.mark.skip(reason="no reference tree at %s" % ref_import.REF_ROOT))
