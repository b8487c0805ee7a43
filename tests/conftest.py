"""pytest configuration: `gpu` marks tests that need a CUDA device (run with -m gpu on a B200)."""
import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); parity tests through the C-ABI")


@pytest.fixture(scope="session")
def H():
    import harness
    return harness


@pytest.fixture(scope="session")
def golden(H):
    return H.golden_vectors()


@pytest.fixture(scope="session")
def small_db(H):
    return H.small_db()


@pytest.fixture(scope="session")
def front_small(H, small_db):
    return H.front.Front(small_db, H.shipped_config(), H.NORM_CSV)


@pytest.fixture(scope="session")
def oracle_small(H, small_db):
    return H.Oracle(small_db)


@pytest.fixture(scope="session")
def reference_small(H, small_db, tmp_path_factory):
    """The compiled reference opened on the small voice (skipped where oracle/_ref is absent)."""
    if not H.have_reference():
        pytest.skip("oracle/_ref not built (reference tree absent)")
    p = tmp_path_factory.mktemp("refdb") / "voice.db"
    p.write_bytes(small_db)
    return H.Reference(str(p))
