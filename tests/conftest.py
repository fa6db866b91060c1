import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "root-simple-mcmc_b200"))
sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def checkers():
    """The CPU checkers, built on demand: the oracle port always; the
    reference-backed one only with REFERENCE=<reference checkout> in the
    environment (otherwise an existing oracle/_ref/libsmcmc_ref.so is used, and
    the tests that need it skip without one)."""
    from oracle import cpu_checkers
    cpu_checkers.build(("orc", "ref"))
    return cpu_checkers


@pytest.fixture(scope="session")
def have_ref(checkers):
    return checkers.available("ref")
