import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def port():
    """The C oracle port (oracle/msm_oracle.c), built on demand with gcc."""
    from oracle import port as p
    p.build()
    return p


@pytest.fixture(scope="session")
def emul():
    """CPU emulation of the product's kernel bodies (tests/emul) — test infrastructure."""
    from tests.emul import harness
    return harness


@pytest.fixture(scope="session")
def bb():
    """The product library, initialised on the GPU."""
    import blitzar_b200 as b
    assert b.sxt_init(num_precomputed_generators=64) == 0
    return b
