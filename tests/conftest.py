import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def oracle_lib():
    from oracle import orc
    orc.build()
    return orc


@pytest.fixture(scope="session")
def reference_lib():
    """oracle/_ref/libsgtd_ref.so: the reference's own STDesc.cpp / cluster_manager.hpp compiled
    against the oracle/shim stand-in headers.  Built from the upstream SGTD sources that
    SGTD_REFERENCE_DIR names, otherwise an already built library is used; skipped if neither is there,
    as those sources are not part of this repository."""
    from oracle import ref
    if not ref.available():
        pytest.skip("needs the upstream SGTD sources: set SGTD_REFERENCE_DIR, or build oracle/_ref")
    ref.lib()
    return ref
