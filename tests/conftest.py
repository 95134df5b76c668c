import os
import sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


@pytest.fixture
def refrec(request):
    """The compiled reference's side of a comparison: live when oracle/_ref is built, else its stored digests (cpulibs.RefRecord)"""
    import re
    import cpulibs
    rec = cpulibs.RefRecord(re.sub(r"[^\w.-]+", "_", request.node.name))
    if not rec.usable():
        pytest.skip(f"neither oracle/_ref nor {os.path.relpath(rec.path, ROOT)}")
    yield rec
    if request.node.stash.get(_CALL_FAILED, False) is False:
        rec.close()


_CALL_FAILED = pytest.StashKey[bool]()


@pytest.hookimpl(wrapper=True)
def pytest_runtest_makereport(item, call):
    rep = yield
    if rep.when == "call":
        item.stash[_CALL_FAILED] = rep.failed
    return rep


@pytest.fixture(scope="session")
def device():
    """The CUDA device handle every gpu test uses; a missing GPU/library is a hard failure, never a skip."""
    import ffmpeg_b200 as fb
    dev = fb.Device(0)
    dev.set_default()
    yield dev
    dev.close()
