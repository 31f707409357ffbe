import os
import sys
from pathlib import Path

import pytest

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))

ORACLE_DIR = REPO / "oracle"
REF_SO = ORACLE_DIR / "_ref" / "libhbref.so"
PORT_SO = ORACLE_DIR / "_ref" / "liboracle_port.so"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _have_gpu():
    try:
        import ctypes
        from handbrake_b200 import LIBHBCU
        lib = ctypes.CDLL(str(LIBHBCU))
        return lib.hbcu_device_count() > 0
    except OSError:
        return False


@pytest.fixture(scope="session")
def ref():
    """the reference's own filters: their stored runs (tests/reference_runs.py); with HBCU_RECORD_REFERENCE=<file> the
    calls run on oracle/_ref/libhbref.so and the stored runs plus every call made are written to <file>"""
    from reference_runs import ReferenceRuns
    out = os.environ.get("HBCU_RECORD_REFERENCE")
    if not out:
        yield ReferenceRuns.load()
        return
    from handbrake_b200.hblib import FilterLib
    if not REF_SO.exists():
        pytest.fail("HBCU_RECORD_REFERENCE is set but oracle/_ref/libhbref.so is not built")
    runs = ReferenceRuns.load(FilterLib(REF_SO))
    yield runs
    runs.save(out)


@pytest.fixture(scope="session")
def cuda_filters():
    import handbrake_b200
    if not _have_gpu():
        pytest.fail("GPU test selected but no CUDA device is visible: there is no CPU fallback")
    return handbrake_b200.filters()
