import os
import sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'opencl-structure-from-motion_b200')
for p in (ROOT, PKG, os.path.join(ROOT, 'oracle')):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a B200 (run on the GPU box with -m gpu)')


@pytest.fixture
def reference(request):
    """Stored outputs of the unmodified reference CPU path for this test (oracle/refgold.py) -- the checker, never the product."""
    import refgold
    return refgold.Reference(request.node.path.stem, request.node.name)


@pytest.fixture(scope='session')
def ctx():
    import visocu_py
    c = visocu_py.Context(0)
    yield c
    c.close()
