import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gr-dvbt2ll_b200", "python"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def compiled_ref():
    """The compiled unmodified reference (oracle/_ref); skip when it was not built (it needs the reference sources,
    which are not part of this repository).  For tests of behaviour only the reference has."""
    from oracle import ref
    if not ref.available():
        pytest.skip("oracle/_ref/libdvbt2ll_ref.so not built (needs the unmodified reference sources at build time)")
    ref.lib().ref_set_quiet(1)
    return ref


@pytest.fixture(scope="session")
def reflib():
    """What the parity tests compare with: the compiled unmodified reference when it was built, else the same block
    API over the numpy oracle (oracle/numpy_ref.py) -- not the reference, but the restatement pinned to the
    reference's stored output (test_oracle_matches_golden) and to a record of its own output for every input the
    tests give it (tests/golden/numpy_ref_ledger.json)."""
    from oracle import ref
    if ref.available():
        ref.lib().ref_set_quiet(1)
        return ref
    from oracle import numpy_ref
    return numpy_ref
