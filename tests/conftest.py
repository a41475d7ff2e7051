import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _ensure_built():
    """The product library is built in-tree; make sure it exists before anything loads it."""
    from sqz_b200 import build
    if build.stale():
        build.build()


_ensure_built()


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    with open(os.path.join(ROOT, "tests", "golden", "golden.json")) as f:
        return json.load(f)["inputs"]


@pytest.fixture(scope="session")
def inputs():
    """name -> uint8 array: the reference tests' synthetic vectors, its six data files and csrc.cat."""
    from sqz_b200 import corpus
    d = {k: np.frombuffer(v, dtype=np.uint8) for k, v in corpus.kat_inputs().items()}
    d.update(corpus.all_files())
    return d


@pytest.fixture(scope="session")
def oracle():
    from oracle import Oracle
    return Oracle.get()


@pytest.fixture(scope="session")
def reference(oracle):
    """The unmodified reference (oracle/_ref) where it was built, else its recorded answers
    (tests/recorded_reference.py)."""
    from oracle import Reference
    if Reference.available() and not os.environ.get("SQZ_RECORD_REFERENCE"):
        yield Reference.get()
        return
    from recorded_reference import RecordedReference
    r = RecordedReference(oracle, record_to=os.environ.get("SQZ_RECORD_REFERENCE"))
    yield r
    r.save()


def fnv(oracle, a) -> str:
    return "%016x" % oracle.fnv(np.ascontiguousarray(a))
