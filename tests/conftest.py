import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run by the driver with -m gpu)")


@pytest.fixture(scope="session")
def b200():
    """The product library bound to cuda:0 (fails loudly when there is no sm_100 device)."""
    import svt_av1_psy_b200 as pkg
    pkg.init(0)
    yield pkg.dsp
    pkg.shutdown()


@pytest.fixture(scope="session")
def oracle():
    import oracle as o
    return o


@pytest.fixture(scope="session")
def refc(oracle):
    """ctypes handle on the unmodified reference objects, for the few tests that exercise the reference library itself
    (they skip where it is not built).  Parity tests take `golden` instead and run everywhere."""
    if oracle.ref is None:
        pytest.skip("oracle/_ref/libsvtav1_ref.so is not built (it needs the reference source tree)")
    return oracle.ref


@pytest.fixture
def golden(request, oracle):
    """tests/reference_golden.py: compares with the live reference where it is built, with its recorded digest everywhere"""
    from reference_golden import Golden
    g = Golden(request.node.path.name + "::" + request.node.name, oracle.ref is not None)
    failed = request.session.testsfailed
    yield g
    if request.session.testsfailed == failed:  # a test that already failed is not reported twice
        g.verify()
