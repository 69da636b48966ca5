import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")
    # Some test modules import the ctypes binding at collection time: in a fresh checkout (built artefacts are not tracked)
    # build before collecting.  A no-op when everything is up to date; on the GPU box the prebuilt files travelled.
    import __graft_entry__ as g
    g.build()


@pytest.fixture(scope="session")
def built():
    """Make sure the native pieces exist (no-op when they are already up to date)."""
    import __graft_entry__ as g
    g.build()
    return True


@pytest.fixture(scope="session")
def orc(built):
    from oracle import loader
    return loader.port()


@pytest.fixture(scope="session")
def _reference(built):
    """The compiled reference (oracle/_ref), or where it is not built the stand-in replaying its recorded results
    (tests/oracle_golden.py).  With ORACLE_GOLDEN_RECORD set, the reference's calls are recorded for that stand-in."""
    import oracle_golden as G
    from oracle import loader
    r = loader.ref()
    if os.environ.get(G.RECORD_ENV):
        if r is None:
            pytest.exit("%s needs oracle/_ref built from the reference tree" % G.RECORD_ENV)
        return G.Record(r, loader.port())
    if r is not None:
        return r
    return G.Replay(loader.port(), G.load_effects())


@pytest.fixture(autouse=True)
def _reference_log(request):
    """Per test: the digest of everything the test asked the reference stand-in must equal the recorded one."""
    import oracle_golden as G
    if "_reference" not in request.fixturenames:
        yield
        return
    o = request.getfixturevalue("_reference")
    if not isinstance(o, G._Oracle):
        yield
        return
    o.log = log = G.new_log(request.node.nodeid)
    log["strict"] = "refo" in request.fixturenames
    yield
    o.log = None
    if isinstance(o, G.Record):
        if log["calls"]:
            G.write_record(os.environ[G.RECORD_ENV], log)
        return
    want = G.load_calls().get(log["test"])
    if log["skipped"] or want is None:
        return
    diff = G.mismatch(log, want)
    assert diff is None, "%s: %s (see tests/oracle_golden.py)" % (log["test"], diff)


@pytest.fixture(scope="session")
def refo(_reference):
    return _reference


@pytest.fixture(scope="session")
def checker(_reference):
    """The strongest CPU checker available: the compiled reference, or its recorded stand-in."""
    return _reference


@pytest.fixture(scope="session")
def gpu(built):
    import libav_b200._lib as L
    L.init(0)
    return L
