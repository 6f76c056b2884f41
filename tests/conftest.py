import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "slow: takes more than a few seconds on CPU")


@pytest.fixture(scope="session")
def oracle_lib():
    from oracle import pyoracle

    pyoracle.build()
    return pyoracle.oracle()


@pytest.fixture(scope="session")
def ref_or_none():
    """the reference's own classes (oracle/_ref) where they are built, else None: tests that take this fixture then
    check against data stored under tests/golden"""
    from oracle import pyoracle

    pyoracle.build()
    return pyoracle.ref() if pyoracle.have_ref() else None


@pytest.fixture(scope="session", autouse=True)
def _built_in_tree():
    """libmalva_gpu.so and malva-geno are built in-tree (git-ignored); make sure they exist and are current before
    any test loads them (a no-op when they are up to date)"""
    from malva_b200 import build as mbuild

    mbuild.build()
