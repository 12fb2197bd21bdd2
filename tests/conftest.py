import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def port_oracle():
    from oracle.oracle_py import PortOracle
    return PortOracle()


@pytest.fixture(scope="session")
def _compiled_ref():
    from oracle.oracle_py import RefOracle
    return RefOracle() if RefOracle.available() else None


@pytest.fixture
def ref_oracle(request, _compiled_ref):
    """The compiled reference (oracle/_ref/libnpref.so) where it is built; elsewhere its answers recorded under
    tests/golden/ref_calls/ (tests/ref_replay.py).  NPH_RECORD_REF=<dir> records them from the compiled reference into <dir>."""
    from tests.ref_replay import ReplayedRef
    record_dir = os.environ.get("NPH_RECORD_REF")
    if record_dir and _compiled_ref is None:
        pytest.fail("NPH_RECORD_REF is set but the compiled reference (oracle/_ref/libnpref.so) is not built")
    if _compiled_ref is not None and not record_dir:
        yield _compiled_ref
        return
    ref = ReplayedRef(request.node, _compiled_ref, record_dir)
    yield ref
    ref.finish()


@pytest.fixture(scope="session")
def engine():
    """One context on cuda:0 through the C ABI. No fallback: a missing library or device is an error."""
    from nanopolish_b200.engine import Engine
    eng = Engine(0)
    yield eng
    eng.close()
