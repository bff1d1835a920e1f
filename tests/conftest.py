import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (an sm_100 GPU)")


@pytest.fixture(scope="session")
def oracle():
    import oracle_lib
    return oracle_lib.load()


@pytest.fixture(scope="session")
def _ref_recordings():
    import recorded_ref
    recorded = {}
    yield recorded
    recorded_ref.save(recorded)


@pytest.fixture
def ref(request, _ref_recordings):
    """The reference's own compiled kernels, replayed from tests/golden/reference/ (recorded_ref.py); with
    JV_RECORD_REFERENCE=1 the library itself, its answers recorded."""
    import oracle_lib
    import recorded_ref
    module, test = request.module.__name__, request.node.name
    if not recorded_ref.RECORD:
        yield recorded_ref.Replay(module, test)
        return
    lib = oracle_lib.load_ref()
    assert lib is not None, "JV_RECORD_REFERENCE=1 needs oracle/_ref/libjvector.so (oracle/build_ref.sh)"
    rec = recorded_ref.Recorder(lib)
    yield rec
    _ref_recordings.setdefault(module, {})[test] = rec.arrays()


@pytest.fixture(scope="session")
def sift():
    import oracle_lib
    return oracle_lib.load_siftsmall()
