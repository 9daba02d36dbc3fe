import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def orc():
    import oracle
    return oracle.Oracle()


@pytest.fixture
def ref(request):
    """The reference's recorded outputs for this test (tests/reference_record.py)."""
    from reference_record import RecordedReference
    return RecordedReference("%s::%s" % (request.node.path.stem, request.node.name))
