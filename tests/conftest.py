import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    from oracle.pyoracle import Oracle, build
    build(ref=None)
    return Oracle()


@pytest.fixture(scope="session")
def ref():
    from oracle.pyoracle import Ref, have_ref
    if not have_ref():
        pytest.skip("oracle/_ref/libcsdr_ref.so not built (set CSDR_REFERENCE to the csdr sources at build time)")
    return Ref()
