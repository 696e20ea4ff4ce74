import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def built():
    """native pieces are built once per session (no-op when up to date)"""
    import __graft_entry__ as ge
    ge.build()
    return True


@pytest.fixture(scope="session")
def orc(built):
    from oracle.oracle import Oracle
    return Oracle("libm")


@pytest.fixture(scope="session")
def orc_pm(built):
    from oracle.oracle import Oracle
    return Oracle("pm")


def pytest_sessionfinish(session, exitstatus):
    from tests import reference_record
    reference_record.save()


@pytest.fixture(scope="session")
def ref_live(built):
    """the reference's compiled transforms themselves, for tests that run them on the reference's own shader tree (their
    results are its source text and are not stored)"""
    from oracle.oracle import Reference
    if not Reference.available():
        pytest.skip("oracle/_ref not built (reference tree absent and no prebuilt copy)")
    return Reference()


@pytest.fixture
def ref(built, request):
    """the reference's compiled transforms (oracle/_ref/libglava_ref.so) where they are built, their recorded results
    elsewhere (tests/reference_record.py)"""
    from oracle.oracle import Reference
    from tests import reference_record
    live = Reference.available()
    return reference_record.ReferenceProxy(reference_record.Session(request, live), Reference() if live else None)


@pytest.fixture
def ref_record(built, request):
    """results of the reference's shader tree (the test module's REF_SHADERS) run through oracle/glsl_interp.py: live
    where the tree is present, recorded elsewhere (tests/reference_record.py)"""
    from tests import reference_record
    return reference_record.Session(request, os.path.isdir(request.module.REF_SHADERS))


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
