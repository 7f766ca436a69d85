import os
import sys
import warnings

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

warnings.filterwarnings("ignore", message=".*use_return_dict.*")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "needs_reference: test imports a checkout of the upstream uoo723/PMGT (oracle/ref_shim.py)")


def _has_cuda():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    from oracle import ref_shim

    have_ref = ref_shim.available()
    have_cuda = _has_cuda()
    for item in items:
        if "needs_reference" in item.keywords and not have_ref:
            item.add_marker(pytest.mark.skip(reason="no checkout of uoo723/PMGT found: set PMGT_REFERENCE_ROOT"))
        if "gpu" in item.keywords and not have_cuda:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))


GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN
