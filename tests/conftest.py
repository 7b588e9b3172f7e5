import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_addoption(parser):
    parser.addoption("--record-reference", action="store_true",
                     help="record what the reference returns to every test using the `ref` fixture into tests/golden/reference_calls.npz "
                          "(needs oracle/_ref/libocvref.so; run it over the CPU tests)")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on a machine with one)")
    config.addinivalue_line("markers", "reference_library: checks the reference library itself against constants kept in the repository; "
                                       "there is nothing to record or replay, it runs only where oracle/_ref is built")


_RECORDED = {}
_REF = []


def pytest_sessionfinish(session):
    if _RECORDED:
        import reference_replay
        reference_replay.save(_RECORDED)


def _port():
    from oracle import build_port
    build_port.build()
    from oracle.api import Oracle
    return Oracle("port")


@pytest.fixture(scope="session")
def port():
    """plain-C restatement of the reference (always available: compiled on demand with gcc)"""
    return _port()


@pytest.fixture()
def ref(request):
    """the unmodified reference built by oracle/build_ref.py; where oracle/_ref is absent, its recorded answers to this test
    (tests/reference_replay.py), and a skip when the test has none"""
    from oracle.api import Oracle, available
    import reference_replay
    test_id = "%s::%s" % (os.path.basename(str(request.node.fspath)), request.node.name)
    if available("ref"):
        if not _REF:
            _REF.append(Oracle("ref"))
        if request.config.getoption("--record-reference") and not request.node.get_closest_marker("reference_library"):
            return reference_replay.Recorder(_REF[0], _port(), _RECORDED, test_id)
        return _REF[0]
    archive = reference_replay.recording()
    if test_id not in archive["tests"]:
        pytest.skip("oracle/_ref/libocvref.so not built and no recording of this test")
    return reference_replay.Replay(archive, archive["tests"][test_id], _port(), test_id)


@pytest.fixture(scope="session")
def oracle():
    """the strongest oracle present: the real reference if built, else the port"""
    from oracle.api import Oracle, available
    return Oracle("ref") if available("ref") else _port()


@pytest.fixture(scope="session")
def cvb():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import opencv_b200 as m
    m.init(0)
    return m


@pytest.fixture()
def rng():
    return np.random.default_rng(0xB200)
