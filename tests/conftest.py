import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle():
    from oracle.binding import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def _refshim_live():
    """The compiled reference (oracle/_ref), or None where it was not built."""
    from oracle.binding import RefShim
    try:
        return RefShim(nocontxt=True, maxres=4096)
    except (FileNotFoundError, OSError):
        return None


@pytest.fixture
def refshim(request):
    """The compiled reference's answers: recorded ones from tests/golden/ref (see tests/refreplay.py), or the live
    reference with HHG_REF_RECORD=<dir> (recording) or for a test without a recording; skips when it has neither."""
    from tests import refreplay
    key = os.path.basename(str(request.node.path)) + "::" + request.node.nodeid.split("::", 1)[1]
    if os.environ.get("HHG_REF_RECORD"):
        live = request.getfixturevalue("_refshim_live")
        if live is None:
            pytest.fail("HHG_REF_RECORD needs the compiled reference (oracle/_ref)")
        sink = {"calls": []}
        yield refreplay.Recorder(live, sink)
        if sink["calls"] is not None and request.node.rep_call.passed:
            if not refreplay.save(key, live.V, sink["calls"], os.environ["HHG_REF_RECORD"]):
                print(f"\n{key}: answers too large to record")
        return
    rec = refreplay.load(key)
    if rec is not None:
        yield refreplay.Replayer(key, *rec)
        return
    live = request.getfixturevalue("_refshim_live")
    if live is None:
        pytest.skip("compiled reference not available (oracle/_ref) and no recorded answers for this test")
    yield live


@pytest.hookimpl(hookwrapper=True)
def pytest_runtest_makereport(item, call):
    rep = (yield).get_result()
    if rep.when == "call":
        item.rep_call = rep


@pytest.fixture(scope="session")
def hhg():
    import hhsuite_b200
    return hhsuite_b200


@pytest.fixture(scope="session")
def gpu_ctx(hhg):
    ctx = hhg.Context()
    yield ctx
    ctx.close()
