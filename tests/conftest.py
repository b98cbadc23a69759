import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


@pytest.fixture(scope="session")
def port():
    from oracle.oracle_py import Port
    return Port()


@pytest.fixture(scope="session")
def shim():
    from oracle.oracle_py import Shim
    return Shim()


@pytest.fixture(scope="session")
def ref(port, shim):
    """The reference build's outputs: the live build where it exists, checked against the records of
    tests/golden/reference_records.json (tests/_recorded_ref.py); DMC_RECORD_REFERENCE=1 rewrites the records."""
    from oracle.oracle_py import Reference
    from _recorded_ref import RecordedReference
    rec = RecordedReference(port, shim, Reference() if Reference.available() else None,
                            record=os.environ.get("DMC_RECORD_REFERENCE") == "1")
    yield rec
    if rec.record:
        rec.save()


@pytest.fixture(scope="session")
def ref_build():
    """The reference build itself, for tests about the build (its sources are not part of the repository)."""
    from oracle.oracle_py import Reference
    if not Reference.available():
        pytest.skip("needs the reference build oracle/_ref/libdmc_ref.so")
    return Reference()
