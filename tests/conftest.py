import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def ref():
    """The unmodified reference (libsecp256k1 + CCAN sha256): its recorded answers (tests/refcalls.py)."""
    from tests import util
    return util.recorded_ref()


@pytest.fixture(scope="session")
def cln():
    """CLN's own plumbing (bitcoin/signature.c, common/node_id.c, gossipd/sigcheck.c), unmodified: its recorded answers."""
    from tests import util
    return util.recorded_cln()


def _live(load):
    try:
        return load()
    except RuntimeError as e:
        pytest.skip(str(e))


@pytest.fixture(scope="session")
def ref_live():
    """The reference library itself, for tests that hand the engine objects it built; skips where oracle/_ref is absent."""
    from tests import util
    return _live(util.load_ref)


@pytest.fixture(scope="session")
def cln_live():
    from tests import util
    return _live(util.load_cln)


@pytest.fixture(scope="session")
def emul():
    from tests import util
    return util.load_emul()


@pytest.fixture(scope="session")
def engine():
    import lightning_b200 as L
    eng = L.SigVerifier(0)
    yield eng
    eng.close()
