import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


@pytest.fixture(scope="session")
def built():
    """Build (or reuse) the product library and the oracle libraries once per session."""
    import __graft_entry__ as g
    g.build()
    return True


@pytest.fixture(scope="session")
def port(built):
    from oracle.pyoracle import Port
    return Port()


@pytest.fixture(scope="session")
def reference_builder(built):
    from oracle.pyoracle import ReferenceBuilder
    if not ReferenceBuilder.available():
        pytest.skip("oracle/_ref builder not built (the reference's source is not present); tests/test_restated_golden.py checks its stored answers")
    return ReferenceBuilder()


@pytest.fixture(scope="session")
def reference_setup(built):
    from oracle.pyoracle import ReferenceSetup
    if not ReferenceSetup.available():
        pytest.skip("oracle/_ref scene set-up not built (the reference's source is not present); tests/test_restated_golden.py checks its stored answers")
    return ReferenceSetup()


@pytest.fixture(scope="session")
def reference(built):
    from oracle.pyoracle import Reference
    if not Reference.available():
        pytest.skip("oracle/_ref not built (the reference's source is not present); tests/test_restated_golden.py checks its stored answers")
    return Reference()
