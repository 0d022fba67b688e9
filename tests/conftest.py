import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "bilevel-gait-gen_b200"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session", autouse=True)
def _build_oracle():
    """The oracle is test infrastructure: build it (and oracle/_ref when BGG_REFERENCE_DIR names the reference's sources) once per session."""
    import pyoracle
    pyoracle.build()
    yield
