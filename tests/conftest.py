import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "needs_reference: needs a tree of the upstream control-pcgrl source "
                                       "(found as oracle/refshim.py finds it)")


def pytest_collection_modifyitems(config, items):
    from oracle import refshim
    have_ref = refshim.available()
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    for item in items:
        if "needs_reference" in item.keywords and not have_ref:
            item.add_marker(pytest.mark.skip(reason="no control-pcgrl reference tree"))
        if "gpu" in item.keywords and not have_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
