import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(autouse=True)
def _recorded_reference(request):
    """each test's calls into the reference library are replayed from its own recording (reference_calls.py)"""
    import reference_calls
    product = None
    if request.node.get_closest_marker("gpu") is not None:
        import finitestateentropy_b200 as fb
        product = fb.lib()
    reference_calls.begin(request.node.nodeid, product)
    yield
    reference_calls.end()
