import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
for p_ in (ROOT, HERE):
    if p_ not in sys.path:
        sys.path.insert(0, p_)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA GPU (B200); run on the GPU box")


@pytest.fixture(autouse=True)
def _replayed_reference_answers_produced():
    """Where the reference's answers are replayed (oracle/ref.py), every array the reference
    wrote must have been produced by the restatement in the same test."""
    yield
    ref = sys.modules.get("oracle.ref")
    missing = ref.unmatched() if ref is not None else []
    assert not missing, "the restatement never produced the reference's recorded arrays of %s" % missing


@pytest.fixture(scope="session")
def ctx():
    import rawspeed_b200 as rs
    c = rs.Context(0)
    yield c
    c.close()
