import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


HAVE_GPU = _have_gpu()


def pytest_collection_modifyitems(config, items):
    if HAVE_GPU:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def pf():
    import pffft_b200
    return pffft_b200


_RECORD_DIR = os.environ.get("PFFFT_B200_RECORD_REFERENCE")
_recording = None


@pytest.fixture
def ref(request):
    """the unmodified reference library built into oracle/_ref (checker only); where it was not built, the plain-C
    restatement with every result checked against the reference's, recorded for this test (oracle/golden.py)"""
    global _recording
    from oracle import golden
    from oracle import ref as R
    key = "%s::%s" % (request.module.__name__, request.node.name)
    if not R.have_ref():
        return golden.checked_restatement(key)
    if _RECORD_DIR:
        if _recording is None:
            _recording = golden.Recording()
        return golden.recording_reference(key, _recording)
    return R.ref()


def pytest_sessionfinish(session, exitstatus):
    if _recording is not None:
        os.makedirs(_RECORD_DIR, exist_ok=True)
        _recording.save(os.path.join(_RECORD_DIR, "reference_samples_%d.npz" % os.getpid()))


@pytest.fixture(scope="session")
def R():
    from oracle import ref as R
    return R


def uniform(rng, n, dtype=np.float32):
    """uniform(-1,1) like the reference validator's frand()*2-1 (benchmarks/bench_pffft.c:318)"""
    return (rng.random(n) * 2 - 1).astype(dtype)
