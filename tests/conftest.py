import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _golden_ref(request, tag, path, load):
    """the compiled reference where it is built, else its recorded answers (tests/refgolden.py)"""
    import refgolden
    m = refgolden.mode(os.path.exists(path))
    if m == "live":
        return load()
    if m == "record":
        request.addfinalizer(refgolden.save)
        return refgolden.GoldenRef(tag, load())
    return refgolden.GoldenRef(tag)


@pytest.fixture(scope="session")
def ref(request):
    """compiled reference CPU path (oracle/_ref), test infrastructure only"""
    import refdirac
    return _golden_ref(request, "ref", refdirac.REF_PATH, refdirac.load)


@pytest.fixture(scope="session")
def refser(request):
    """the compiled reference with the worker threads of its robust RTR / NSD solvers run
    synchronously (oracle/ref_shim_rtr_serial.c): deterministic pin of solver_mode 5 and 6"""
    import refdirac
    return _golden_ref(request, "refser", refdirac.SERIAL_PATH, refdirac.load_serial)


@pytest.fixture(scope="session")
def api():
    """the product library; GPU tests only"""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sagecal_b200 import lib
    return lib.load()
