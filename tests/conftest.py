import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle.reference_cases import random_graph_edges  # noqa: E402,F401  (seeded edge lists, shared with the record)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    with open(os.path.join(ROOT, "tests", "golden", "golden.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def orc():
    """The CPU oracle (test infrastructure; see oracle/oracle.cpp)."""
    from oracle import binding
    binding.build()
    return binding.oracle()


@pytest.fixture(scope="session")
def ref_or_none():
    """The reference library where it is present, else None: tests that compare with it then use the stored record."""
    from oracle import binding
    return binding.reference()


@pytest.fixture(scope="session")
def reference_cases():
    """What the reference answers on the seeded cases of the CPU suite (oracle/reference_cases.py)."""
    from oracle import reference_cases
    return reference_cases.load()


@pytest.fixture(scope="session")
def gms():
    """The product (CUDA through the C ABI)."""
    import gms_b200
    gms_b200.lib()
    return gms_b200
