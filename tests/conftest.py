import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run on the GPU box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    """The CPU oracle (test infrastructure; oracle/plstvo_oracle.c)."""
    from oracle.oracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def engine():
    """The CUDA library through its C-ABI.  Fails loudly when the extension or the GPU is missing."""
    from stvo_pl_b200.engine import Engine
    return Engine()


@pytest.fixture
def ref(request):
    """The reference's own pose code (oracle/_ref), as recorded for this test in tests/golden/ref_outputs.npz."""
    import ref_golden
    return ref_golden.for_test(request.node)


GOLDEN = os.path.join(ROOT, "tests", "golden")
