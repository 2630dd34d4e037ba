import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _ensure_built():
    import __graft_entry__ as ge
    ge.build()


@pytest.fixture(scope="session")
def zq():
    _ensure_built()
    import zpaqfranz_b200
    return zpaqfranz_b200


@pytest.fixture(scope="session")
def ctx(zq):
    c = zq.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="session")
def oracle():
    """oracle/_ref/libzqoracle.so -- this repo's plain-C restatement (the checker)."""
    _ensure_built()
    import oracle_bindings
    return oracle_bindings.load_oracle()


@pytest.fixture(scope="session")
def ref():
    """The reference's answers (checker): recorded under tests/golden/ref/.  With ZQ_RECORD_REF=<dir> set, the reference
    itself (oracle/_ref/libzpaqref.so), every answer written to <dir>/<test module>.json at the end of the session."""
    import oracle_bindings
    out = os.environ.get("ZQ_RECORD_REF")
    if not out:
        yield oracle_bindings.GoldenRef()
        return
    _ensure_built()
    r = oracle_bindings.load_ref()
    assert r is not None, "ZQ_RECORD_REF needs the reference: oracle/_ref/libzpaqref.so is not built"
    rec = oracle_bindings.RecordingRef(r)
    yield rec
    rec.save(out)
