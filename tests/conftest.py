import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.dirname(os.path.abspath(__file__))):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def pkg():
    import rte_b200

    return rte_b200.pkg


@pytest.fixture(scope="session")
def oracle_port():
    import oraclelib

    return oraclelib.load("port")


@pytest.fixture(scope="session")
def oracle_ref():
    import oraclelib

    if not oraclelib.have_ref():
        pytest.skip("oracle/_ref not built: build() makes it where it finds the original project's source "
                    "(ORE_REFERENCE_DIR, see oracle/ref_build/make_ref.py)")
    return oraclelib.load("ref")


@pytest.fixture(scope="session")
def oracle_best():
    import oraclelib

    return oraclelib.load("best")


@pytest.fixture(scope="session")
def renderer(pkg):
    """One context on cuda:0 through the C ABI; fails loudly (no fallback) if unusable."""
    pkg.build.build_library()
    r = pkg.Renderer(0)
    yield r
    r.close()
