import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


def _has_gpu():
    try:
        from directxtex_b200 import capi
        return capi.lib.dxb200_device_count() > 0
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def oracle():
    """The reference's answers (tests/golden/reference_calls.npz).  With DXB_RECORD_REFERENCE=<file> the calls go to the
    reference build instead (oracle/_ref/libdxtex_ref.so, oracle/Makefile) and are recorded into <file> at the end of the session."""
    from tests import oracle_lib
    ref = oracle_lib.load_reference_answers()
    yield ref
    if isinstance(ref, oracle_lib.Recorder):
        ref.save(os.environ["DXB_RECORD_REFERENCE"])


@pytest.fixture(scope="session")
def emul():
    from tests import oracle_lib
    return oracle_lib.load_emul()
